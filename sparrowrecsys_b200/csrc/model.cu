// model.cu - the C ABI (include/srs_ctr.h): model construction (validation + the private
// device re-layout of the reference's weights), and the predict entry points.
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <initializer_list>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/srs_ctr.h"
#include "kernels.h"

namespace srs {
cudaError_t setup_embmlp_attributes();
cudaError_t setup_deepfm_attributes();
cudaError_t setup_din_attributes();
cudaError_t setup_dien_attributes();
cudaError_t setup_din_tc_attributes();
cudaError_t setup_din_rt_attributes();
cudaError_t setup_din_rtp_attributes();
cudaError_t setup_din_rt64_attributes();
cudaError_t setup_embmlp_tc_attributes();
cudaError_t setup_deepfm_tc_attributes();
// gather.cu
struct PeerGather;
cudaError_t gather_create(int device, int world, int rank, int64_t slice_rows, PeerGather** out);
cudaError_t gather_export(PeerGather* g, void* handle64);
cudaError_t gather_connect(PeerGather* g, const void* handles);
void gather_destroy(PeerGather* g);
bool gather_connected(const PeerGather* g);
int gather_begin_step(PeerGather* g, BatchView& v, bool in_kernel_signal);
cudaError_t gather_signal(PeerGather* g, cudaStream_t s);
cudaError_t gather_wait(PeerGather* g, cudaStream_t s);
float* gather_buffer(PeerGather* g, int parity);
int gather_parity(const PeerGather* g);
int64_t gather_rows(const PeerGather* g);
int gather_device(const PeerGather* g);
int64_t gather_slice_rows(const PeerGather* g);
}  // namespace srs

using namespace srs;

namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

}  // namespace

namespace srs {
// srs_last_error() of the entry points defined outside this file (retrieve.cu)
int report_error(int code, const char* msg) { return fail(code, "%s", msg); }
}  // namespace srs

namespace {

// Kernel-variant options of the model being created: "key=value;key=value" handed to
// srs_model_create_ex (keys: din_impl, embmlp_impl, deepfm_impl, zero_copy_scores).  The environment variables SRS_<KEY> remain as a tuning override of last resort.
thread_local std::string g_create_opts;
const char* opt(const char* key, const char* env_name) {
  static thread_local std::string val;
  const std::string& o = g_create_opts;
  const std::string k = std::string(key) + "=";
  size_t pos = 0;
  while (pos < o.size()) {
    size_t end = o.find(';', pos);
    if (end == std::string::npos) end = o.size();
    if (o.compare(pos, k.size(), k) == 0) {
      val = o.substr(pos + k.size(), end - pos - k.size());
      return val.c_str();
    }
    pos = end + 1;
  }
  return getenv(env_name);
}

#define CUDA_TRY(expr)                                                                   \
  do {                                                                                   \
    cudaError_t e__ = (expr);                                                            \
    if (e__ != cudaSuccess)                                                              \
      return fail(SRS_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), \
                  __FILE__, __LINE__);                                                   \
  } while (0)

constexpr int kSlots = 4;           // public pipelining slots; slot kSlots is private to
                                    // the synchronous srs_predict_host
constexpr int kErrWords = kSlots + 2;

struct Slot {
  cudaStream_t stream = nullptr;
  int capacity = 0;                 // rows the device staging can hold
  uint8_t* d_block = nullptr;       // one allocation: [movie|user|hist|movie_genre|user_genre|numerics]
  float* d_probs = nullptr;
  float* d_logits = nullptr;
  int32_t* d_hist32 = nullptr;      // widened history ids when the batch came with hist16
  int rank_capacity = 0;            // srs_rank_host only: rows d_rank can rank
  uint8_t* d_rank = nullptr;        // [top_idx cap | top_scores cap | sort scratch]
  int* h_err = nullptr;             // pinned mirror of the device error flag
  // latency path (synchronous single calls): the last kernel of the call writes {sequence number, error
  // word} into a pinned record the caller spins on - no device-to-host copy, no stream synchronise
  uint32_t* h_done = nullptr;       // pinned [4]
  uint32_t seq = 0;
  int res_capacity = 0;
  int32_t* h_res = nullptr;         // pinned: top positions [cap] | top scores [cap]
  int req_capacity = 0;             // srs_rank_user_host only: candidates the request staging holds
  int32_t* d_req = nullptr;         // [user row | history | candidate ids] on the device
  int32_t* h_req = nullptr;         // pinned copy of it
};

// The forward kernel a model runs, chosen when it is created.  din_rt, din_rtp and din_rt64 all read
// srs_model::din_rt.
enum class Kernel { ncf, embmlp, embmlp_tc, deepfm, deepfm_tc, deepfm2, din, din_tc, din_rt, din_rtp, din_rt64, dien };

}  // namespace

struct srs_model {
  srs_spec spec{};
  int device = 0;
  int EP = 0;
  int hist_cols = 0;                // history columns the model reads (T for DIN, 1 for W&D)
  bool dense_feats = false;         // reads movie_genre / user_genre / numerics (all but NeuralCF and two towers)
  std::vector<void*> owned;
  int* err_flag = nullptr;          // kErrWords device words: [0] srs_predict_device, [1 + i] host slot i.  One word
                                    // per slot: a flag shared by every slot could be copied by slot A, set by
                                    // slot B's kernel and cleared by A's wait before B ever read it
  NcfParams ncf{};
  EmbMlpParams emb{};
  DeepFmParams fm{};
  DeepFm2Params fm2{};
  DinParams din{};
  DienParams dien{};
  DinTcParams din_tc{};
  DinRtParams din_rt{};
  EmbMlpTcParams emb_tc{};
  DeepFmTcParams fm_tc{};
  Kernel kernel = Kernel::ncf;
  bool no_zero_copy = false;         // SRS_ZERO_COPY_SCORES=0 switches the latency path of srs_predict_host off
  bool zero_copy_scores = false;     // SRS_ZERO_COPY_SCORES=1 (experimental): kernels write the scores
                                     // of a host batch straight into the caller's pinned buffer
  void* movie_feats = nullptr;       // srs_model_set_movie_features: [n][8 words] movie-side features in HBM
  int movie_feats_rows = 0;
  int device_sms = 148;
  int64_t bytes_per_inf = 0;
  Slot slots[kSlots + 1];
  std::mutex mu;
};

namespace {
inline int* slot_err(srs_model* m, const Slot& s) { return m->err_flag + 1 + (&s - m->slots); }

const char* kernel_name(const srs_model* m) {
  const bool wide = m->spec.kind == SRS_WIDENDEEP;
  switch (m->kernel) {
    case Kernel::ncf: return m->spec.kind == SRS_TWOTOWERS ? "ncf_kernel<two_towers>" : "ncf_kernel<neural_cf_model_1>";
    case Kernel::embmlp: return wide ? "embmlp_kernel<wide&deep>" : "embmlp_kernel";
    case Kernel::embmlp_tc: return wide ? "embmlp_tc_kernel<wide&deep>" : "embmlp_tc_kernel";
    case Kernel::deepfm: return "deepfm_kernel";
    case Kernel::deepfm_tc: return "deepfm_tc_kernel";
    case Kernel::deepfm2: return "deepfm2_kernel";
    case Kernel::din: return "din_kernel";
    case Kernel::din_tc: return "din_tc_kernel";
    case Kernel::din_rt: return "din_rt_kernel";
    case Kernel::din_rtp: return "din_rtp_kernel";
    case Kernel::din_rt64: return "din_rt64_kernel";
    case Kernel::dien: return "dien_kernel";
  }
  return "";
}

// A kernel the `*_impl` option can force: the option value, whether the model's shape fits the kernel, and
// the error when it is forced onto a shape that does not.
struct Forced {
  const char* value;
  Kernel kernel;
  bool fits;
  const char* needs;
};

// m->kernel = `def`, unless the create option `key` (else the environment variable `env`) names one of
// `forced`; a value that names none of them leaves the default.
int select_kernel(srs_model* m, const char* key, const char* env, Kernel def, std::initializer_list<Forced> forced) {
  m->kernel = def;
  const char* impl = opt(key, env);
  if (!impl) return SRS_OK;
  for (const Forced& f : forced)
    if (!strcmp(impl, f.value)) {
      if (!f.fits) return fail(SRS_ERR_INVALID, "%s", f.needs);
      m->kernel = f.kernel;
    }
  return SRS_OK;
}
}  // namespace


namespace {

int round_ep(int E) {
  if (E <= 12) return 12;
  if (E <= 16) return 16;
  if (E <= 32) return 32;
  return 64;
}

struct Builder {
  srs_model* m;
  std::map<std::string, const srs_tensor*> by_name;
  int status = SRS_OK;

  const srs_tensor* need(const char* name, int64_t rows, int64_t cols) {
    if (status != SRS_OK) return nullptr;
    auto it = by_name.find(name);
    if (it == by_name.end()) {
      status = fail(SRS_ERR_MISSING, "missing weight tensor '%s'", name);
      return nullptr;
    }
    const srs_tensor* t = it->second;
    if (t->rows != rows || t->cols != cols) {
      status = fail(SRS_ERR_SHAPE, "weight '%s' has shape [%lld,%lld], expected [%lld,%lld]", name,
                    (long long)t->rows, (long long)t->cols, (long long)rows, (long long)cols);
      return nullptr;
    }
    if (t->data == nullptr) {
      status = fail(SRS_ERR_INVALID, "weight '%s' has a null data pointer", name);
      return nullptr;
    }
    return t;
  }

  // dense host tensor -> float vector (must be SRS_HOST)
  const float* host(const char* name, int64_t rows, int64_t cols) {
    const srs_tensor* t = need(name, rows, cols);
    if (!t) return nullptr;
    if (t->location != SRS_HOST) {
      status = fail(SRS_ERR_INVALID, "weight '%s' must be a host tensor", name);
      return nullptr;
    }
    return t->data;
  }

  // device allocation owned by the model
  void* alloc(size_t bytes) {
    if (status != SRS_OK) return nullptr;
    void* d = nullptr;
    cudaError_t e = cudaMalloc(&d, bytes);
    if (e != cudaSuccess) {
      status = fail(SRS_ERR_NOMEM, "cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
      return nullptr;
    }
    m->owned.push_back(d);
    return d;
  }

  template <class T>
  T* upload(const std::vector<T>& v) {
    T* d = static_cast<T*>(alloc((v.size() ? v.size() : 1) * sizeof(T)));
    if (d && !v.empty()) {
      cudaError_t e = cudaMemcpy(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice);
      if (e != cudaSuccess) {
        status = fail(SRS_ERR_CUDA, "cudaMemcpy H2D failed: %s", cudaGetErrorString(e));
        return nullptr;
      }
    }
    return d;
  }

  // embedding table [V][E] -> device [V][EP] (zero padded rows), chunked upload
  const float* table(const char* name, int64_t V, int E) {
    const srs_tensor* t = need(name, V, E);
    if (!t) return nullptr;
    const int EP = m->EP;
    if (t->location == SRS_DEVICE_BORROWED) {
      if (E != EP) {
        status = fail(SRS_ERR_INVALID,
                      "borrowed device table '%s' needs emb_dim == padded dim (%d != %d)", name, E, EP);
        return nullptr;
      }
      return t->data;
    }
    float* d = nullptr;
    size_t bytes = (size_t)V * EP * sizeof(float);
    cudaError_t e = cudaMalloc(&d, bytes);
    if (e != cudaSuccess) {
      status = fail(SRS_ERR_NOMEM, "cudaMalloc(%zu) for '%s' failed: %s", bytes, name,
                    cudaGetErrorString(e));
      return nullptr;
    }
    m->owned.push_back(d);
    if (E == EP) {
      e = cudaMemcpy(d, t->data, bytes, cudaMemcpyHostToDevice);
    } else {
      const int64_t chunk = 1 << 16;
      std::vector<float> buf((size_t)std::min<int64_t>(chunk, V) * EP);
      e = cudaSuccess;
      for (int64_t v0 = 0; v0 < V && e == cudaSuccess; v0 += chunk) {
        const int64_t nv = std::min<int64_t>(chunk, V - v0);
        std::fill(buf.begin(), buf.end(), 0.f);
        for (int64_t v = 0; v < nv; ++v)
          memcpy(&buf[(size_t)v * EP], t->data + (size_t)(v0 + v) * E, (size_t)E * sizeof(float));
        e = cudaMemcpy(d + (size_t)v0 * EP, buf.data(), (size_t)nv * EP * sizeof(float),
                       cudaMemcpyHostToDevice);
      }
    }
    if (e != cudaSuccess) {
      status = fail(SRS_ERR_CUDA, "table upload '%s' failed: %s", name, cudaGetErrorString(e));
      return nullptr;
    }
    return d;
  }

  // Dense kernel [K][N] -> [dev_rows][NP]: device row i takes reference row map[i]
  // (-1 = zero row); columns zero padded to NP.
  std::vector<float> permute(const float* ref, int N, const std::vector<int>& map, int NP) {
    std::vector<float> out(map.size() * (size_t)NP, 0.f);
    if (!ref) return out;
    for (size_t i = 0; i < map.size(); ++i)
      if (map[i] >= 0)
        for (int j = 0; j < N; ++j) out[i * NP + j] = ref[(size_t)map[i] * N + j];
    return out;
  }

  std::vector<float> padvec(const float* ref, int n, int np) {
    std::vector<float> out(np, 0.f);
    if (ref)
      for (int i = 0; i < n; ++i) out[i] = ref[i];
    return out;
  }
};

std::vector<int> iota_map(int start, int n, int padded) {
  std::vector<int> v(padded, -1);
  for (int i = 0; i < n; ++i) v[i] = start + i;
  return v;
}

void append(std::vector<int>& a, const std::vector<int>& b) { a.insert(a.end(), b.begin(), b.end()); }

// Rows of a reference layer-1 dense/kernel: the first row of each embedding block, in the order the
// kernels gather the blocks, and the seven numeric rows in NUMERIC_KEYS order.
struct DenseRows {
  std::vector<int> emb;
  int num[7];
};

// DenseFeatures sorted concat (SURVEY.md 8a row a2): movieGenre1..3, movieId, userGenre1..5, userId
DenseRows embmlp_rows(int E) {
  return {{1, 1 + E, 1 + 2 * E, 1 + 3 * E, 5 + 4 * E, 5 + 5 * E, 5 + 6 * E, 5 + 7 * E, 5 + 8 * E, 5 + 9 * E},
          {0, 1 + 4 * E, 2 + 4 * E, 3 + 4 * E, 4 + 4 * E, 5 + 10 * E, 6 + 10 * E}};
}

// deep movieId, deep userId
DenseRows deepfm_rows(int E) { return {{1, 5 + E}, {0, 1 + E, 2 + E, 3 + E, 4 + E, 5 + 2 * E, 6 + 2 * E}}; }

// [user_profile | pooled | candidate | context] (DIN.py:161-162): userGenre1, userId, pooled behaviours,
// candidate, movieGenre1
DenseRows din_rows(int E) {
  const int base = 3 + 4 * E;
  return {{1, 1 + E, 3 + 2 * E, 3 + 3 * E, base + 1},
          {base, base + 1 + E, base + 2 + E, base + 3 + E, 0, 1 + 2 * E, 2 + 2 * E}};
}

// CUDA-core layer-1 row map: every embedding block padded to EP, then the numerics and one zero row
std::vector<int> layer1_map(const DenseRows& r, int E, int EP) {
  std::vector<int> map;
  for (int start : r.emb) append(map, iota_map(start, E, EP));
  map.insert(map.end(), r.num, r.num + 7);
  map.push_back(-1);
  return map;
}

// [8][pitch] numeric rows of layer 1 (row 7 zero), the fp32 term of the tensor-core kernels
std::vector<float> pack_w1num(const float* k1, int h0, const DenseRows& r, int pitch) {
  std::vector<float> w((size_t)8 * pitch, 0.f);
  for (int n = 0; n < 7; ++n)
    for (int j = 0; j < h0; ++j) w[(size_t)n * pitch + j] = k1[(size_t)r.num[n] * h0 + j];
  return w;
}

// ------------------------------------------------------------------------------------
int build_ncf(Builder& B) {
  srs_model* m = B.m;
  const srs_spec& s = m->spec;
  const int E = s.emb_dim, EP = m->EP;
  const bool two = s.kind == SRS_TWOTOWERS;
  if (s.n_hidden < 1 || s.n_hidden > 3) return fail(SRS_ERR_INVALID, "1..3 hidden layers supported");
  int hmax = 0;
  for (int i = 0; i < s.n_hidden; ++i) hmax = std::max(hmax, s.hidden[i]);
  if (hmax > 32 || hmax < 1) return fail(SRS_ERR_INVALID, "hidden widths must be in 1..32");
  const int HP = hmax <= 16 ? 16 : 32;
  NcfParams& p = m->ncf;
  p.movie = B.table("movieId_embedding", s.n_movies, E);
  p.user = B.table("userId_embedding", s.n_users, E);
  p.n_movies = s.n_movies; p.n_users = s.n_users;
  p.EP = EP; p.HP = HP; p.n_layers = s.n_hidden; p.two_towers = two; p.final_dense = s.final_dense;
  std::vector<float> blob;
  auto push = [&](const std::vector<float>& v) {
    int off = (int)blob.size();
    blob.insert(blob.end(), v.begin(), v.end());
    while (blob.size() % 4) blob.push_back(0.f);
    return off;
  };
  char name[64];
  if (!two) {
    int in = 2 * E;
    for (int l = 0; l < s.n_hidden; ++l) {
      const int out = s.hidden[l];
      snprintf(name, sizeof(name), "dense_%d/kernel", l);
      const float* k = B.host(name, in, out);
      snprintf(name, sizeof(name), "dense_%d/bias", l);
      const float* bias = B.host(name, out, 1);
      std::vector<int> map;
      if (l == 0) { append(map, iota_map(0, E, EP)); append(map, iota_map(E, E, EP)); }
      else map = iota_map(0, in, HP);
      p.w_off[l] = push(B.permute(k, out, map, HP));
      p.b_off[l] = push(B.padvec(bias, out, HP));
      in = out;
    }
    snprintf(name, sizeof(name), "dense_%d/kernel", s.n_hidden);
    const float* k = B.host(name, in, 1);
    snprintf(name, sizeof(name), "dense_%d/bias", s.n_hidden);
    const float* bias = B.host(name, 1, 1);
    p.out_w = push(B.padvec(k, in, HP));
    p.out_b = push(B.padvec(bias, 1, 4));
  } else {
    const char* sides[2] = {"item", "user"};
    for (int t = 0; t < 2; ++t) {
      int in = E;
      for (int l = 0; l < s.n_hidden; ++l) {
        const int out = s.hidden[l];
        snprintf(name, sizeof(name), "%s_dense_%d/kernel", sides[t], l);
        const float* k = B.host(name, in, out);
        snprintf(name, sizeof(name), "%s_dense_%d/bias", sides[t], l);
        const float* bias = B.host(name, out, 1);
        std::vector<int> map = l == 0 ? iota_map(0, E, EP) : iota_map(0, in, HP);
        p.w_off[3 * t + l] = push(B.permute(k, out, map, HP));
        p.b_off[3 * t + l] = push(B.padvec(bias, out, HP));
        in = out;
      }
    }
    if (s.final_dense) {
      const float* k = B.host("dense_out/kernel", 1, 1);
      const float* bias = B.host("dense_out/bias", 1, 1);
      p.out_w = push(B.padvec(k, 1, 4));
      p.out_b = push(B.padvec(bias, 1, 4));
    } else {
      p.out_w = push(std::vector<float>(4, 1.f));
      p.out_b = push(std::vector<float>(4, 0.f));
    }
  }
  if (B.status != SRS_OK) return B.status;
  p.blob = B.upload(blob);
  p.blob_floats = (int)blob.size();
  return B.status;
}

int build_embmlp(Builder& B) {
  srs_model* m = B.m;
  const srs_spec& s = m->spec;
  const int E = s.emb_dim, EP = m->EP;
  const bool wide = s.kind == SRS_WIDENDEEP;
  if (s.n_hidden != 2 || s.hidden[0] > 128 || s.hidden[1] > 128 || s.hidden[0] < 1 || s.hidden[1] < 1)
    return fail(SRS_ERR_INVALID, "EmbeddingMLP/W&D need two hidden layers of width <= 128");
  const int h0 = s.hidden[0], h1 = s.hidden[1];
  EmbMlpParams& p = m->emb;
  char name[64];
  for (int k = 0; k < 3; ++k) {
    snprintf(name, sizeof(name), "movieGenre%d_embedding", k + 1);
    p.genre[k] = B.table(name, s.n_genres, E);
  }
  for (int k = 0; k < 5; ++k) {
    snprintf(name, sizeof(name), "userGenre%d_embedding", k + 1);
    p.genre[3 + k] = B.table(name, s.n_genres, E);
  }
  p.movie = B.table("movieId_embedding", s.n_movies, E);
  p.user = B.table("userId_embedding", s.n_users, E);
  const float* k1 = B.host("dense/kernel", 7 + 10 * E, h0);
  const float* b1 = B.host("dense/bias", h0, 1);
  const float* k2 = B.host("dense_1/kernel", h0, h1);
  const float* b2 = B.host("dense_1/bias", h1, 1);
  const int last_in = h1 + (wide ? s.cross_buckets : 0);
  const float* k3 = B.host("dense_2/kernel", last_in, 1);
  const float* b3 = B.host("dense_2/bias", 1, 1);
  if (B.status != SRS_OK) return B.status;
  p.W1 = B.upload(B.permute(k1, h0, layer1_map(embmlp_rows(E), E, EP), 128));
  p.b1 = B.upload(B.padvec(b1, h0, 128));
  p.W2 = B.upload(B.permute(k2, h1, iota_map(0, h0, 128), 128));
  p.b2 = B.upload(B.padvec(b2, h1, 128));
  p.w3 = B.upload(B.padvec(k3, h1, 128));
  p.wide = nullptr;
  if (wide) p.wide = B.upload(std::vector<float>(k3 + h1, k3 + h1 + s.cross_buckets));
  p.b3 = b3[0];
  p.n_movies = s.n_movies; p.n_users = s.n_users; p.n_genres = s.n_genres;
  p.cross_buckets = s.cross_buckets; p.EP = EP;
  return B.status;
}

int build_deepfm(Builder& B) {
  srs_model* m = B.m;
  const srs_spec& s = m->spec;
  const int E = s.emb_dim, EP = m->EP;
  if (s.n_hidden != 2 || s.hidden[0] > 64 || s.hidden[1] > 64 || s.hidden[0] < 1 || s.hidden[1] < 1)
    return fail(SRS_ERR_INVALID, "DeepFM needs two hidden layers of width <= 64");
  const int h0 = s.hidden[0], h1 = s.hidden[1];
  const int64_t fm1 = (int64_t)2 * s.n_genres + s.n_movies + s.n_users;
  DeepFmParams& p = m->fm;
  p.fm_movie = B.table("fm_movieId_embedding", s.n_movies, E);
  p.fm_user = B.table("fm_userId_embedding", s.n_users, E);
  p.fm_mgenre = B.table("fm_movieGenre1_embedding", s.n_genres, E);
  p.fm_ugenre = B.table("fm_userGenre1_embedding", s.n_genres, E);
  p.deep_movie = B.table("deep_movieId_embedding", s.n_movies, E);
  p.deep_user = B.table("deep_userId_embedding", s.n_users, E);
  const float* k1 = B.host("dense/kernel", 7 + 2 * E, h0);
  const float* b1 = B.host("dense/bias", h0, 1);
  const float* k2 = B.host("dense_1/kernel", h0, h1);
  const float* b2 = B.host("dense_1/bias", h1, 1);
  const float* k3 = B.host("dense_2/kernel", fm1 + 4 + h1, 1);
  const float* b3 = B.host("dense_2/bias", 1, 1);
  if (B.status != SRS_OK) return B.status;
  p.W1 = B.upload(B.permute(k1, h0, layer1_map(deepfm_rows(E), E, EP), 64));
  p.b1 = B.upload(B.padvec(b1, h0, 64));
  p.W2 = B.upload(B.permute(k2, h1, iota_map(0, h0, 64), 64));
  p.b2 = B.upload(B.padvec(b2, h1, 64));
  p.first = B.upload(std::vector<float>(k3, k3 + fm1));
  for (int d = 0; d < 4; ++d) p.wdot[d] = k3[fm1 + d];
  p.wdeep = B.upload(B.padvec(k3 + fm1 + 4, h1, 64));
  p.bout = b3[0];
  p.n_movies = s.n_movies; p.n_users = s.n_users; p.n_genres = s.n_genres; p.EP = EP;
  return B.status;
}

int build_deepfm2(Builder& B) {
  srs_model* m = B.m;
  const srs_spec& s = m->spec;
  const int E = s.emb_dim, EP = m->EP, P = 64;
  if (s.proj_dim != P) return fail(SRS_ERR_INVALID, "DeepFM_v2 projection width must be 64");
  if (s.n_hidden != 2 || s.hidden[0] > 32 || s.hidden[1] > 16 || s.hidden[0] < 1 || s.hidden[1] < 1)
    return fail(SRS_ERR_INVALID, "DeepFM_v2 needs hidden widths <= (32, 16)");
  const int h0 = s.hidden[0], h1 = s.hidden[1];
  const int64_t fm1 = (int64_t)2 * s.n_genres + s.n_movies + s.n_users;
  DeepFm2Params& p = m->fm2;
  p.mgenre = B.table("movieGenre1_embedding", s.n_genres, E);
  p.movie = B.table("movieId_embedding", s.n_movies, E);
  p.ugenre = B.table("userGenre1_embedding", s.n_genres, E);
  p.user = B.table("userId_embedding", s.n_users, E);
  const float* fc = B.host("first_cat/kernel", fm1, 1);
  const float* fcb = B.host("first_cat/bias", 1, 1);
  const float* fn = B.host("first_num/kernel", 7, 1);
  const float* fnb = B.host("first_num/bias", 1, 1);
  const char* fields[4] = {"movieGenre1", "movieId", "userGenre1", "userId"};
  const float* pk[4]; const float* pb[4];
  char name[64];
  for (int f = 0; f < 4; ++f) {
    snprintf(name, sizeof(name), "proj_%s/kernel", fields[f]);
    pk[f] = B.host(name, E, P);
    snprintf(name, sizeof(name), "proj_%s/bias", fields[f]);
    pb[f] = B.host(name, P, 1);
  }
  const float* pnk = B.host("proj_num/kernel", 7, P);
  const float* pnb = B.host("proj_num/bias", P, 1);
  const float* dk = B.host("deep/kernel", 5 * P, h0);
  const float* db = B.host("deep/bias", h0, 1);
  const float* d1k = B.host("deep_1/kernel", h0, h1);
  const float* d1b = B.host("deep_1/bias", h1, 1);
  const float* ok = B.host("out/kernel", 1 + P + h1, 1);
  const float* ob = B.host("out/bias", 1, 1);
  if (B.status != SRS_OK) return B.status;
  p.first = B.upload(std::vector<float>(fc, fc + fm1));
  p.first_num = B.upload(B.padvec(fn, 7, 8));
  p.first_bias = fcb[0] + fnb[0];
  for (int f = 0; f < 4; ++f) {
    p.proj[f] = B.upload(B.permute(pk[f], P, iota_map(0, E, EP), P));
    p.proj_b[f] = B.upload(B.padvec(pb[f], P, P));
  }
  p.proj_num = B.upload(B.permute(pnk, P, iota_map(0, 7, 8), P));
  p.proj_num_b = B.upload(B.padvec(pnb, P, P));
  p.Wd = B.upload(B.permute(dk, h0, iota_map(0, 5 * P, 5 * P), 32));
  p.bd = B.upload(B.padvec(db, h0, 32));
  p.Wd1 = B.upload(B.permute(d1k, h1, iota_map(0, h0, 32), 16));
  p.bd1 = B.upload(B.padvec(d1b, h1, 16));
  p.wout = B.upload(B.padvec(ok, 1 + P + h1, 1 + P + 16));
  p.bout = ob[0];
  p.n_movies = s.n_movies; p.n_users = s.n_users; p.n_genres = s.n_genres; p.EP = EP;
  return B.status;
}

int build_din(Builder& B) {
  srs_model* m = B.m;
  const srs_spec& s = m->spec;
  const int E = s.emb_dim, EP = m->EP, T = s.hist_len, A = 32;
  if (s.au_hidden != A) return fail(SRS_ERR_INVALID, "DIN activation-unit width must be 32");
  if (s.n_hidden != 2 || s.hidden[0] > 128 || s.hidden[1] > 64 || s.hidden[0] < 1 || s.hidden[1] < 1)
    return fail(SRS_ERR_INVALID, "DIN needs hidden widths <= (128, 64)");
  if (T < 1) return fail(SRS_ERR_INVALID, "hist_len must be >= 1");
  const int h0 = s.hidden[0], h1 = s.hidden[1];
  DinParams& p = m->din;
  p.movie = B.table("embedding", s.n_movies, E);
  p.user = B.table("userId_embedding", s.n_users, E);
  p.ugenre = B.table("userGenre1_embedding", s.n_genres, E);
  p.mgenre = B.table("movieGenre1_embedding", s.n_genres, E);
  const float* au = B.host("au_dense/kernel", 4 * E, A);
  const float* aub = B.host("au_dense/bias", A, 1);
  const float* alpha = B.host("au_prelu/alpha", T, A);
  const float* auo = B.host("au_out/kernel", A, 1);
  const float* auob = B.host("au_out/bias", 1, 1);
  const float* k1 = B.host("dense/kernel", 5 * E + 7, h0);
  const float* b1 = B.host("dense/bias", h0, 1);
  const float* a1 = B.host("prelu/alpha", h0, 1);
  const float* k2 = B.host("dense_1/kernel", h0, h1);
  const float* b2 = B.host("dense_1/bias", h1, 1);
  const float* a2 = B.host("prelu_1/alpha", h1, 1);
  const float* k3 = B.host("dense_2/kernel", h1, 1);
  const float* b3 = B.host("dense_2/bias", 1, 1);
  if (B.status != SRS_OK) return B.status;
  // activation-unit fold: rows of au_dense/kernel are [h-c | h | c | h*c] blocks of E
  std::vector<float> wh((size_t)EP * A, 0.f), wp((size_t)EP * A, 0.f), wc((size_t)EP * A, 0.f);
  for (int e = 0; e < E; ++e)
    for (int j = 0; j < A; ++j) {
      const float w_sub = au[(size_t)e * A + j], w_h = au[(size_t)(E + e) * A + j];
      const float w_c = au[(size_t)(2 * E + e) * A + j], w_p = au[(size_t)(3 * E + e) * A + j];
      wh[(size_t)e * A + j] = w_sub + w_h;
      wp[(size_t)e * A + j] = w_p;
      wc[(size_t)e * A + j] = w_c - w_sub;
    }
  p.au_wh = B.upload(wh); p.au_wp = B.upload(wp); p.au_wc = B.upload(wc);
  p.au_b = B.upload(std::vector<float>(aub, aub + A));
  p.au_alpha = B.upload(std::vector<float>(alpha, alpha + (size_t)T * A));
  p.au_wout = B.upload(std::vector<float>(auo, auo + A));
  p.au_bout = auob[0];
  p.W1 = B.upload(B.permute(k1, h0, layer1_map(din_rows(E), E, EP), 128));
  p.b1 = B.upload(B.padvec(b1, h0, 128));
  p.a1 = B.upload(B.padvec(a1, h0, 128));
  p.W2 = B.upload(B.permute(k2, h1, iota_map(0, h0, 128), 64));
  p.b2 = B.upload(B.padvec(b2, h1, 64));
  p.a2 = B.upload(B.padvec(a2, h1, 64));
  p.w3 = B.upload(B.padvec(k3, h1, 64));
  p.b3 = b3[0];
  p.n_movies = s.n_movies; p.n_users = s.n_users; p.n_genres = s.n_genres;
  p.T = T; p.EP = EP;
  return B.status;
}

// ---- DIEN (DIEN.py:154-256): sequence-part blob in the layout of dien.cu::DienBlob<EP> ---------
int build_dien(Builder& B) {
  srs_model* m = B.m;
  const srs_spec& s = m->spec;
  const int E = s.emb_dim, EP = m->EP, T = s.hist_len, A = 32;
  if (E > 32) return fail(SRS_ERR_INVALID, "DIEN supports emb_dim <= 32");
  if (s.au_hidden != A) return fail(SRS_ERR_INVALID, "DIEN attention width must be 32");
  if (s.n_hidden != 2 || s.hidden[0] > 128 || s.hidden[1] > 64 || s.hidden[0] < 1 || s.hidden[1] < 1)
    return fail(SRS_ERR_INVALID, "DIEN needs hidden widths <= (128, 64)");
  if (T < 1) return fail(SRS_ERR_INVALID, "hist_len must be >= 1");
  const int h0 = s.hidden[0], h1 = s.hidden[1];
  DienParams& p = m->dien;
  p.movie = B.table("embedding", s.n_movies, E);
  p.user = B.table("userId_embedding", s.n_users, E);
  p.ugenre = B.table("userGenre1_embedding", s.n_genres, E);
  p.mgenre = B.table("movieGenre1_embedding", s.n_genres, E);
  const float* gk = B.host("gru/kernel", E, 3 * E);
  const float* gr = B.host("gru_recurrent/kernel", E, 3 * E);
  const float* gb = B.host("gru/bias", 2, 3 * E);
  const float* ak = B.host("att_dense/kernel", E, A);
  const float* ab = B.host("att_dense/bias", A, 1);
  const float* ao = B.host("att_out/kernel", A, 1);
  const float* aob = B.host("att_out/bias", 1, 1);
  const char* gates[3] = {"r", "z", "h"};
  const float *wi[3], *bi[3], *wh[3], *wa[3], *ba[3];
  for (int g = 0; g < 3; ++g) {
    char name[64];
    snprintf(name, sizeof name, "augru_%s_input/kernel", gates[g]); wi[g] = B.host(name, E, E);
    snprintf(name, sizeof name, "augru_%s_input/bias", gates[g]); bi[g] = B.host(name, E, 1);
    snprintf(name, sizeof name, "augru_%s_hidden/kernel", gates[g]); wh[g] = B.host(name, E, E);
    snprintf(name, sizeof name, "augru_%s_act/kernel", gates[g]); wa[g] = B.host(name, E, E);
    snprintf(name, sizeof name, "augru_%s_act/bias", gates[g]); ba[g] = B.host(name, E, 1);
  }
  const float* u0 = B.host("augru_h0", 1, E);
  const float* k1 = B.host("dense/kernel", 5 * E + 7, h0);
  const float* b1 = B.host("dense/bias", h0, 1);
  const float* a1 = B.host("prelu/alpha", h0, 1);
  const float* k2 = B.host("dense_1/kernel", h0, h1);
  const float* b2 = B.host("dense_1/bias", h1, 1);
  const float* a2 = B.host("prelu_1/alpha", h1, 1);
  const float* k3 = B.host("dense_2/kernel", h1, 1);
  const float* b3 = B.host("dense_2/bias", 1, 1);
  if (B.status != SRS_OK) return B.status;
  const int total = dien_seq_floats(EP);
  if (total < 0) return fail(SRS_ERR_INVALID, "DIEN: unsupported padded width %d", EP);
  std::vector<float> q((size_t)total, 0.f);
  const int EE = EP * EP;
  const int GW = 0, GU = 3 * EE, AW = 6 * EE, IW = AW + 32 * EP, HW = IW + 3 * EE, SW = HW + 3 * EE,
            BX = SW + 3 * EE, BH = BX + 3 * EP, BI = BH + 3 * EP, BA = BI + 3 * EP, H0 = BA + 3 * EP,
            AB = H0 + EP, AO = AB + 32, ABO = AO + 32;
  for (int k = 0; k < E; ++k)
    for (int g = 0; g < 3; ++g)                 // Keras gate blocks z | r | h along the 3E axis
      for (int e = 0; e < E; ++e) {
        q[GW + (size_t)k * 3 * EP + g * EP + e] = gk[(size_t)k * 3 * E + g * E + e];
        q[GU + (size_t)k * 3 * EP + g * EP + e] = gr[(size_t)k * 3 * E + g * E + e];
      }
  for (int g = 0; g < 3; ++g)
    for (int e = 0; e < E; ++e) {
      q[BX + g * EP + e] = gb[g * E + e];
      q[BH + g * EP + e] = gb[3 * E + g * E + e];
      q[BI + g * EP + e] = bi[g][e];
      q[BA + g * EP + e] = ba[g][e];
    }
  for (int k = 0; k < E; ++k)
    for (int j = 0; j < A; ++j) q[AW + (size_t)k * 32 + j] = ak[(size_t)k * A + j];
  for (int g = 0; g < 3; ++g)
    for (int k = 0; k < E; ++k)
      for (int e = 0; e < E; ++e) {
        q[IW + (size_t)g * EE + k * EP + e] = wi[g][(size_t)k * E + e];
        q[HW + (size_t)g * EE + k * EP + e] = wh[g][(size_t)k * E + e];
        q[SW + (size_t)g * EE + k * EP + e] = wa[g][(size_t)k * E + e];
      }
  for (int e = 0; e < E; ++e) q[H0 + e] = u0[e];
  for (int j = 0; j < A; ++j) { q[AB + j] = ab[j]; q[AO + j] = ao[j]; }
  q[ABO] = aob[0];
  p.seq = B.upload(q);
  // top kernel rows: [augru | candidate | user_profile | context] (DIEN.py:250); the blocks
  // are DenseFeatures layers, sorted by column name inside (as in DIN)
  // embedding blocks in DIN's gather order: userGenre1, userId, AUGRU final state, candidate, movieGenre1
  const int up = 2 * E, ctx = 4 * E + 3;
  const DenseRows rows = {{up + 1, up + 1 + E, 0, E, ctx + 1},
                          {ctx, ctx + 1 + E, ctx + 2 + E, ctx + 3 + E, up, up + 1 + 2 * E, up + 2 + 2 * E}};
  p.W1 = B.upload(B.permute(k1, h0, layer1_map(rows, E, EP), 128));
  p.b1 = B.upload(B.padvec(b1, h0, 128));
  p.a1 = B.upload(B.padvec(a1, h0, 128));
  p.W2 = B.upload(B.permute(k2, h1, iota_map(0, h0, 128), 64));
  p.b2 = B.upload(B.padvec(b2, h1, 64));
  p.a2 = B.upload(B.padvec(a2, h1, 64));
  p.w3 = B.upload(B.padvec(k3, h1, 64));
  p.b3 = b3[0];
  p.n_movies = s.n_movies; p.n_users = s.n_users; p.n_genres = s.n_genres;
  p.T = T; p.EP = EP;
  return B.status;
}

// ---- tensor-core DIN: shared-memory image ------------------------------------------------
inline uint32_t f2u(float x) { uint32_t u; memcpy(&u, &x, 4); return u; }
inline float u2f(uint32_t u) { float x; memcpy(&x, &u, 4); return x; }
inline uint16_t bf16_rn_bits(float x) {
  const uint32_t u = f2u(x);
  return (uint16_t)((u + 0x7FFFu + ((u >> 16) & 1u)) >> 16);
}
inline uint32_t sw128_off(uint32_t row, uint32_t chunk) { return row * 128u + ((chunk ^ (row & 7u)) << 4); }

// Write logical matrix M[rows][64*kblocks] (via getter) as K-major SW128 bf16 tiles; `part`
// selects the hi half (x rounded to bf16) or the lo half (x - hi rounded to bf16).
template <class F>
void write_sw128(uint8_t* dst, int rows, int kblocks, bool lo_part, F get) {
  for (int kb = 0; kb < kblocks; ++kb)
    for (int r = 0; r < rows; ++r)
      for (int c = 0; c < 8; ++c)
        for (int i = 0; i < 8; ++i) {
          const float x = get(r, kb * 64 + c * 8 + i);
          const uint16_t hb = bf16_rn_bits(x);
          const uint16_t v = lo_part ? bf16_rn_bits(x - u2f((uint32_t)hb << 16)) : hb;
          memcpy(dst + (size_t)kb * rows * 128 + sw128_off(r, c) + i * 2, &v, 2);
        }
}

// Layer-1 embedding weights as hi and lo MMA operands: row = unit j, K = block * width + e, the blocks of
// `r.emb` in order (zero for j >= h0, e >= E and past the last block).
void write_w1_image(uint8_t* hi, uint8_t* lo, int kblocks, const float* k1, int h0, const DenseRows& r, int E,
                    int width) {
  const int nb = (int)r.emb.size();
  auto get = [&](int j, int k) -> float {
    const int b = k / width, e = k - b * width;
    if (j >= h0 || b >= nb || e >= E) return 0.f;
    return k1[(size_t)(r.emb[b] + e) * h0 + j];
  };
  write_sw128(hi, 128, kblocks, false, get);
  write_sw128(lo, 128, kblocks, true, get);
}

// Layer-2 weights W2^T [unit i][k], zero for i >= h1 or k >= h0
float w2t(const float* k2, int h0, int h1, int i, int k) { return (i < h1 && k < h0) ? k2[(size_t)k * h1 + i] : 0.f; }

void write_w2_image(uint8_t* hi, uint8_t* lo, int kblocks, const float* k2, int h0, int h1) {
  auto get = [&](int i, int k) { return w2t(k2, h0, h1, i, k); };
  write_sw128(hi, 128, kblocks, false, get);
  write_sw128(lo, 128, kblocks, true, get);
}

// DIN's layer-2 A operand, one 128-row tile per K block: rows 0..63 = hi halves of W2^T, rows 64..127 = lo halves
void write_w2_stacked(uint8_t* dst, const float* k2, int h0, int h1) {
  for (int kb = 0; kb < 2; ++kb)
    for (int r = 0; r < 128; ++r)
      for (int c = 0; c < 8; ++c)
        for (int i = 0; i < 8; ++i) {
          const float x = w2t(k2, h0, h1, r & 63, kb * 64 + c * 8 + i);
          const uint16_t hb = bf16_rn_bits(x);
          const uint16_t v = (r < 64) ? hb : bf16_rn_bits(x - u2f((uint32_t)hb << 16));
          memcpy(dst + (size_t)kb * 16384 + sw128_off(r, c) + i * 2, &v, 2);
        }
}

// Activation unit, history side: (Wsub + Wh)^T and Wp^T as [unit j][e] with row pitch `pitch`, zero beyond E
// (rows of au_dense/kernel are [h-c | h | c | h*c] blocks of E)
void au_transposed(const float* au, int E, int pitch, std::vector<float>& waT, std::vector<float>& wpT) {
  const int A = 32;
  waT.assign((size_t)A * pitch, 0.f);
  wpT.assign((size_t)A * pitch, 0.f);
  for (int j = 0; j < A; ++j)
    for (int e = 0; e < E; ++e) {
      waT[(size_t)j * pitch + e] = au[(size_t)e * A + j] + au[(size_t)(E + e) * A + j];
      wpT[(size_t)j * pitch + e] = au[(size_t)(3 * E + e) * A + j];
    }
}

// PReLU + Dense(1) of the activation unit folded into two tables per position t < T:
//   wout_j max(v,0) + alpha_tj wout_j min(v,0) = v P_tj + |v| Q_tj;  put(t, j, P_tj, Q_tj)
template <class F>
void fold_pq(const float* alpha, const float* auo, int T, F put) {
  for (int t = 0; t < T; ++t)
    for (int j = 0; j < 32; ++j) {
      const float wo = auo[j], aw = alpha[(size_t)t * 32 + j] * auo[j];
      put(t, j, 0.5f * (wo + aw), 0.5f * (wo - aw));
    }
}

// Tables and vectors build_din uploaded (or borrowed) that the tensor-core DIN kernels read unchanged
template <class P>
void copy_din_common(P& p, const DinParams& v1) {
  p.movie = v1.movie; p.user = v1.user; p.ugenre = v1.ugenre; p.mgenre = v1.mgenre;
  p.au_wc = v1.au_wc; p.au_b = v1.au_b;
  p.b1 = v1.b1; p.a1 = v1.a1;
  p.b2 = v1.b2; p.a2 = v1.a2; p.w3 = v1.w3;
  p.au_bout = v1.au_bout; p.b3 = v1.b3;
  p.n_movies = v1.n_movies; p.n_users = v1.n_users; p.n_genres = v1.n_genres;
  p.T = v1.T;
}

// Fills m->din_tc from the same reference tensors build_din validated.
int build_din_tc(Builder& B) {
  srs_model* m = B.m;
  const srs_spec& s = m->spec;
  const int E = s.emb_dim, T = s.hist_len, A = 32;
  const int h0 = s.hidden[0], h1 = s.hidden[1];
  const int CPR = (T + 31) / 32, TP = CPR * 32;
  const float* au = B.host("au_dense/kernel", 4 * E, A);
  const float* alpha = B.host("au_prelu/alpha", T, A);
  const float* auo = B.host("au_out/kernel", A, 1);
  const float* k1 = B.host("dense/kernel", 5 * E + 7, h0);
  const float* k2 = B.host("dense_1/kernel", h0, h1);
  if (B.status != SRS_OK) return B.status;
  const DenseRows rows = din_rows(E);
  // image offsets mirror the constants in din_tc.cu
  const uint32_t IMG_AUB_HI = 0, IMG_AUB_LO = 4096, IMG_W1_HI = 8192, IMG_W1_LO = IMG_W1_HI + 3 * 16384,
                 IMG_W2 = IMG_W1_LO + 3 * 16384, IMG_PQ = IMG_W2 + 2 * 16384;
  const uint32_t kPqStride = 68;
  std::vector<uint8_t> img(IMG_PQ + (uint32_t)TP * kPqStride * 4u, 0);
  // activation unit B operand: row j = [ (Wsub+Wh)[e][j], e<32 | Wp[e][j], e<32 ]
  std::vector<float> waT, wpT;
  au_transposed(au, E, 32, waT, wpT);
  auto au_get = [&](int j, int k) -> float { return (k < 32 ? waT : wpT)[(size_t)j * 32 + (k & 31)]; };
  write_sw128(img.data() + IMG_AUB_HI, 32, 1, false, au_get);
  write_sw128(img.data() + IMG_AUB_LO, 32, 1, true, au_get);
  // layer 1 A operand: row = unit j, K = [userGenre1 | userId | pooled | candidate | movieGenre1 | 0] x 32
  write_w1_image(img.data() + IMG_W1_HI, img.data() + IMG_W1_LO, 3, k1, h0, rows, E, 32);
  write_w2_stacked(img.data() + IMG_W2, k2, h0, h1);
  // P/Q: one 68-float row per position t (zero beyond T), stored as 16 x (P_2m, P_2m+1, Q_2m, Q_2m+1) so
  // one 128-bit load feeds two packed FMAs
  float* PQ = reinterpret_cast<float*>(img.data() + IMG_PQ);
  fold_pq(alpha, auo, T, [&](int t, int j, float P, float Q) {
    float* cell = PQ + (size_t)t * kPqStride + (j >> 1) * 4 + (j & 1);
    cell[0] = P;
    cell[2] = Q;
  });
  DinTcParams& p = m->din_tc;
  copy_din_common(p, m->din);
  p.image = B.upload(img);
  p.w1num = B.upload(pack_w1num(k1, h0, rows, 128));
  for (int j = 0; j < A; ++j) p.au_wout[j] = auo[j];
  p.CPR = CPR;
  p.num_sms = m->device_sms;
  return B.status;
}

// Row-tile DIN kernels, E padded to 32 (din_rt.cu; din_rtp.cu runs the same parameters) or to 64
// (din_rt64.cu): pre-split movie table, transposed activation-unit weights, P/Q gate tables and the
// top-MLP operand images, from the tensors build_din validated.
int build_din_rt(Builder& B) {
  srs_model* m = B.m;
  const srs_spec& s = m->spec;
  const int E = s.emb_dim, EP = m->EP, T = s.hist_len, A = 32;
  const int h0 = s.hidden[0], h1 = s.hidden[1];
  const float* au = B.host("au_dense/kernel", 4 * E, A);
  const float* alpha = B.host("au_prelu/alpha", T, A);
  const float* auo = B.host("au_out/kernel", A, 1);
  const float* k1 = B.host("dense/kernel", 5 * E + 7, h0);
  const float* k2 = B.host("dense_1/kernel", h0, h1);
  if (B.status != SRS_OK) return B.status;
  const DenseRows rows = din_rows(E);
  // operand images: W1 has one EP-wide K slot per embedding block (3 or 5 K blocks of 16 KB); the order is
  // W2 | W1 hi | W1 lo in din_rt.cu and W1 hi | W1 lo | W2 in din_rt64.cu
  const uint32_t w1_blocks = EP == 32 ? 3 : 5, w1_bytes = w1_blocks * 16384, w2_bytes = 2 * 16384;
  const uint32_t W1_HI = EP == 32 ? w2_bytes : 0, W1_LO = W1_HI + w1_bytes, W2 = EP == 32 ? 0 : 2 * w1_bytes;
  std::vector<uint8_t> img(2 * w1_bytes + w2_bytes, 0);
  write_w1_image(img.data() + W1_HI, img.data() + W1_LO, w1_blocks, k1, h0, rows, E, EP);
  write_w2_stacked(img.data() + W2, k2, h0, h1);
  std::vector<float> waT, wpT;
  au_transposed(au, E, EP, waT, wpT);
  std::vector<float> pq((size_t)T * 64, 0.f);          // [T][P_t 32 | Q_t 32]
  fold_pq(alpha, auo, T, [&](int t, int j, float P, float Q) {
    pq[(size_t)t * 64 + j] = P;
    pq[(size_t)t * 64 + 32 + j] = Q;
  });
  DinRtParams& p = m->din_rt;
  copy_din_common(p, m->din);
  p.image = B.upload(img);
  // history rows: [n_movies][EP bf16 hi | EP bf16 lo]
  void* d_split = B.alloc((size_t)s.n_movies * EP * 4);
  if (B.status != SRS_OK) return B.status;
  const cudaError_t e = EP == 32 ? launch_split_table(m->din.movie, d_split, s.n_movies, nullptr)
                                 : launch_split_table64(m->din.movie, d_split, s.n_movies, nullptr);
  if (e != cudaSuccess) return fail(SRS_ERR_CUDA, "table split failed: %s", cudaGetErrorString(e));
  p.movie_split = static_cast<const uint8_t*>(d_split);
  p.waT = B.upload(waT); p.wpT = B.upload(wpT); p.pq = B.upload(pq);
  p.w1num = B.upload(pack_w1num(k1, h0, rows, 128));
  p.rows_per_group = 32;
  if (EP == 64) p.nch = T > 128 ? 2 : 1;
  p.num_sms = m->device_sms;
  if (m->kernel != Kernel::din_rtp) return B.status;
  // din_rtp: W1^T over K = [userId | pooled | candidate] as a tensor-memory A operand (lane = unit, one 32-bit
  // column per pair of consecutive k: 48 hi words, then 48 lo words), and the two genre blocks of dense/kernel
  // folded into fp32 tables G[genre][unit] = emb[genre] . rows (exact: 19 values)
  std::vector<uint32_t> w1t_words((size_t)128 * 96, 0u);
  auto w1k = [&](int j, int k) -> float {
    const int f = k >> 5, ee = k & 31;
    if (j >= h0 || ee >= E) return 0.f;
    return k1[(size_t)(rows.emb[1 + f] + ee) * h0 + j];
  };
  for (int j = 0; j < 128; ++j)
    for (int w = 0; w < 48; ++w) {
      uint32_t hi = 0, lo = 0;
      for (int half = 0; half < 2; ++half) {
        const float x = w1k(j, 2 * w + half);
        const uint16_t hb = bf16_rn_bits(x);
        const uint16_t lb = bf16_rn_bits(x - u2f((uint32_t)hb << 16));
        hi |= (uint32_t)hb << (16 * half);
        lo |= (uint32_t)lb << (16 * half);
      }
      w1t_words[(size_t)j * 96 + w] = hi;
      w1t_words[(size_t)j * 96 + 48 + w] = lo;
    }
  const float* ug = B.host("userGenre1_embedding", s.n_genres, E);
  const float* mg = B.host("movieGenre1_embedding", s.n_genres, E);
  if (B.status != SRS_OK) return B.status;
  std::vector<float> gtab_u((size_t)s.n_genres * 128, 0.f), gtab_m((size_t)s.n_genres * 128, 0.f);
  for (int g = 0; g < s.n_genres; ++g)
    for (int j = 0; j < h0; ++j) {
      double su = 0.0, sm = 0.0;
      for (int ee = 0; ee < E; ++ee) {
        su += (double)ug[(size_t)g * E + ee] * (double)k1[(size_t)(rows.emb[0] + ee) * h0 + j];
        sm += (double)mg[(size_t)g * E + ee] * (double)k1[(size_t)(rows.emb[4] + ee) * h0 + j];
      }
      gtab_u[(size_t)g * 128 + j] = (float)su;
      gtab_m[(size_t)g * 128 + j] = (float)sm;
    }
  p.w1_tmem = B.upload(w1t_words);
  p.gtab_u = B.upload(gtab_u);
  p.gtab_m = B.upload(gtab_m);
  const cudaError_t ea = setup_din_rtp_attributes();
  if (ea != cudaSuccess) return fail(SRS_ERR_CUDA, "din_rtp attribute setup failed: %s", cudaGetErrorString(ea));
  return B.status;
}

// Tensor-core EmbeddingMLP / W&D (E <= 12): operand images from the tensors build_embmlp validated.
int build_embmlp_tc(Builder& B) {
  srs_model* m = B.m;
  const srs_spec& s = m->spec;
  const int E = s.emb_dim, h0 = s.hidden[0], h1 = s.hidden[1];
  const float* k1 = B.host("dense/kernel", 7 + 10 * E, h0);
  const float* k2 = B.host("dense_1/kernel", h0, h1);
  if (B.status != SRS_OK) return B.status;
  const DenseRows rows = embmlp_rows(E);
  std::vector<uint8_t> img(131072, 0);
  write_w1_image(img.data() + 0, img.data() + 32768, 2, k1, h0, rows, E, 12);     // K = block * 12 + e
  write_w2_image(img.data() + 65536, img.data() + 98304, 2, k2, h0, h1);
  EmbMlpTcParams& p = m->emb_tc;
  const EmbMlpParams& v1 = m->emb;
  for (int k = 0; k < 8; ++k) p.genre[k] = v1.genre[k];
  p.movie = v1.movie; p.user = v1.user;
  p.image = B.upload(img);
  p.b1 = v1.b1; p.b2 = v1.b2; p.w3 = v1.w3; p.wide = v1.wide; p.b3 = v1.b3;
  p.w1num = B.upload(pack_w1num(k1, h0, rows, 128));
  p.n_movies = s.n_movies; p.n_users = s.n_users; p.n_genres = s.n_genres; p.cross_buckets = s.cross_buckets;
  p.num_sms = m->device_sms;
  return B.status;
}

// Tensor-core DeepFM (emb_dim 13..16): operand images from the tensors build_deepfm validated.
int build_deepfm_tc(Builder& B) {
  srs_model* m = B.m;
  const srs_spec& s = m->spec;
  const int E = s.emb_dim, h0 = s.hidden[0], h1 = s.hidden[1];
  const float* k1 = B.host("dense/kernel", 7 + 2 * E, h0);
  const float* k2 = B.host("dense_1/kernel", h0, h1);
  if (B.status != SRS_OK) return B.status;
  const DenseRows rows = deepfm_rows(E);
  std::vector<uint8_t> img(65536, 0);
  write_w1_image(img.data() + 0, img.data() + 16384, 1, k1, h0, rows, E, 16);     // K = [movieId 16 | userId 16 | 0]
  write_w2_image(img.data() + 32768, img.data() + 49152, 1, k2, h0, h1);
  DeepFmTcParams& p = m->fm_tc;
  const DeepFmParams& v1 = m->fm;
  p.fm_movie = v1.fm_movie; p.fm_user = v1.fm_user; p.fm_mgenre = v1.fm_mgenre; p.fm_ugenre = v1.fm_ugenre;
  p.deep_movie = v1.deep_movie; p.deep_user = v1.deep_user;
  p.image = B.upload(img);
  p.b1 = v1.b1; p.b2 = v1.b2; p.first = v1.first; p.wdeep = v1.wdeep;
  p.w1num = B.upload(pack_w1num(k1, h0, rows, 64));
  for (int d = 0; d < 4; ++d) p.wdot[d] = v1.wdot[d];
  p.bout = v1.bout;
  p.n_movies = s.n_movies; p.n_users = s.n_users; p.n_genres = s.n_genres;
  p.num_sms = m->device_sms;
  return B.status;
}

int64_t bytes_per_inference(const srs_spec& s) {
  const int64_t E = s.emb_dim, T = s.hist_len;
  switch (s.kind) {
    case SRS_EMBEDDINGMLP: return 10 * 4 * E + 10 * 4 + 7 * 4 + 4;
    case SRS_WIDENDEEP: return 10 * 4 * E + 11 * 4 + 7 * 4 + 4 + 4;
    case SRS_NEURALCF:
    case SRS_TWOTOWERS: return 2 * 4 * E + 2 * 4 + 4;
    case SRS_DEEPFM: return 6 * 4 * E + 4 * 4 + 4 * 4 + 7 * 4 + 4;
    case SRS_DEEPFM_V2: return 4 * 4 * E + 4 * 4 + 4 * 4 + 7 * 4 + 4;
    case SRS_DIN:
    case SRS_DIEN: return (T + 1) * 4 * E + 3 * 4 * E + 28 + 4 * (T + 4) + 4;
  }
  return 0;
}

int check_batch(const srs_model* m, const srs_batch* b) {
  if (!m || !b) return fail(SRS_ERR_INVALID, "null model or batch");
  if (b->B < 0) return fail(SRS_ERR_INVALID, "negative batch size");
  if (b->B == 0) return SRS_OK;
  if (!b->movie_id || !b->user_id) return fail(SRS_ERR_INVALID, "movie_id / user_id are required");
  if (m->dense_feats && (!b->movie_genre || !b->user_genre || !b->numerics))
    return fail(SRS_ERR_INVALID, "movie_genre / user_genre / numerics are required for this model");
  if (m->hist_cols > 0) {
    if (!b->hist && !b->hist16) return fail(SRS_ERR_INVALID, "hist is required for this model");
    if (b->hist16 && m->spec.n_movies > 65536)
      return fail(SRS_ERR_INVALID, "hist16 needs a movie vocabulary of at most 65536 ids");
    if (b->hist_stride < m->hist_cols)
      return fail(SRS_ERR_INVALID, "hist_stride %d < history columns %d", b->hist_stride, m->hist_cols);
  }
  return SRS_OK;
}

int launch(srs_model* m, const BatchView& v, cudaStream_t stream) {
  cudaError_t e = cudaSuccess;
  switch (m->kernel) {
    case Kernel::ncf: e = launch_ncf(m->ncf, v, stream); break;
    case Kernel::embmlp: e = launch_embmlp(m->emb, v, stream); break;
    case Kernel::embmlp_tc: e = launch_embmlp_tc(m->emb_tc, v, stream); break;
    case Kernel::deepfm: e = launch_deepfm(m->fm, v, stream); break;
    case Kernel::deepfm_tc: e = launch_deepfm_tc(m->fm_tc, v, stream); break;
    case Kernel::deepfm2: e = launch_deepfm2(m->fm2, v, stream); break;
    case Kernel::din: e = launch_din(m->din, v, stream); break;
    case Kernel::din_tc: e = launch_din_tc(m->din_tc, v, stream); break;
    case Kernel::din_rt: e = launch_din_rt(m->din_rt, v, stream); break;
    case Kernel::din_rtp: e = launch_din_rtp(m->din_rt, v, stream); break;
    case Kernel::din_rt64: e = launch_din_rt64(m->din_rt, v, stream); break;
    case Kernel::dien: e = launch_dien(m->dien, v, stream); break;
  }
  if (e != cudaSuccess) return fail(SRS_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
  return SRS_OK;
}

// Device staging of one batch is a single block in the canonical packed order
//   [movie_id B | user_id B | hist B*hc | movie_genre B*3 | user_genre B*5 | numerics B*7] x 4 bytes;
// a host batch laid out the same way (arrays back to back) goes over PCIe as ONE copy.
struct PackedLayout {
  size_t movie, user, hist, mg, ug, num, total;
};
PackedLayout packed_layout(const srs_model* m, size_t B, bool narrow_hist = false) {
  const bool dense_feats = m->dense_feats;
  PackedLayout L{};
  size_t off = 0;
  L.movie = off; off += B * 4;
  L.user = off; off += B * 4;
  L.hist = off;
  off += narrow_hist ? ((B * (size_t)m->hist_cols * 2 + 3) & ~(size_t)3) : B * (size_t)m->hist_cols * 4;
  L.mg = off; off += dense_feats ? B * 3 * 4 : 0;
  L.ug = off; off += dense_feats ? B * 5 * 4 : 0;
  L.num = off; off += dense_feats ? B * 7 * 4 : 0;
  L.total = off;
  return L;
}

// Kernel view of a batch staged at `d` in the packed order; the caller sets the outputs and the error word.
BatchView packed_view(const srs_model* m, const uint8_t* d, const PackedLayout& L, int B) {
  BatchView v{};
  v.B = B; v.hist_stride = m->hist_cols;
  v.movie_id = reinterpret_cast<const int32_t*>(d + L.movie);
  v.user_id = reinterpret_cast<const int32_t*>(d + L.user);
  v.hist = reinterpret_cast<const int32_t*>(d + L.hist);
  v.movie_genre = reinterpret_cast<const int32_t*>(d + L.mg);
  v.user_genre = reinterpret_cast<const int32_t*>(d + L.ug);
  v.numerics = reinterpret_cast<const float*>(d + L.num);
  return v;
}

// Kernel view of a batch whose arrays are on the device already (after check_batch); the caller sets the
// outputs.
int device_view(srs_model* m, const srs_batch* b, BatchView& v) {
  if (m->hist_cols > 0 && !b->hist)
    return fail(SRS_ERR_INVALID, "device batches carry int32 history ids (hist16 is for host batches)");
  CUDA_TRY(cudaSetDevice(m->device));
  v = BatchView{};
  v.B = b->B; v.hist_stride = b->hist_stride;
  v.movie_id = b->movie_id; v.user_id = b->user_id; v.hist = b->hist;
  v.movie_genre = b->movie_genre; v.user_genre = b->user_genre; v.numerics = b->numerics;
  v.err_flag = m->err_flag;
  return SRS_OK;
}

int ensure_slot(srs_model* m, Slot& s, int B) {
  if (!s.stream) CUDA_TRY(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
  if (!s.h_err) {
    CUDA_TRY(cudaMallocHost(&s.h_err, sizeof(int)));
    *s.h_err = 0;
  }
  if (B <= s.capacity) return SRS_OK;
  int cap = std::max(B, 1024);
  cudaFree(s.d_block); cudaFree(s.d_probs); cudaFree(s.d_logits); cudaFree(s.d_hist32);
  s.d_block = nullptr; s.d_probs = nullptr; s.d_logits = nullptr; s.d_hist32 = nullptr;
  s.capacity = 0;
  CUDA_TRY(cudaMalloc(&s.d_block, packed_layout(m, (size_t)cap).total + 256));
  CUDA_TRY(cudaMalloc(&s.d_probs, (size_t)cap * 4));
  CUDA_TRY(cudaMalloc(&s.d_logits, (size_t)cap * 4));
  if (m->hist_cols > 0 && m->spec.n_movies <= 65536)
    CUDA_TRY(cudaMalloc(&s.d_hist32, (size_t)cap * m->hist_cols * 4));
  s.capacity = cap;
  return SRS_OK;
}

// H2D of the batch into the slot's staging and the forward kernel, on the slot's stream;
// the scores are left in s.d_probs (and s.d_logits).
// `probs_out`: where the kernel writes the scores (default: the slot's device buffer).
int stage_and_launch(srs_model* m, Slot& s, const srs_batch* b, bool want_logits,
                     float* probs_out = nullptr, float* logits_out = nullptr) {
  int rc = check_batch(m, b);
  if (rc != SRS_OK) return rc;
  CUDA_TRY(cudaSetDevice(m->device));
  rc = ensure_slot(m, s, b->B);
  if (rc != SRS_OK) return rc;
  if (b->B == 0) return SRS_OK;
  const size_t B = (size_t)b->B;
  const bool narrow = m->hist_cols > 0 && b->hist16 != nullptr;
  const PackedLayout L = packed_layout(m, B, narrow);
  uint8_t* d = s.d_block;
  const uint8_t* h0 = reinterpret_cast<const uint8_t*>(b->movie_id);
  bool packed = reinterpret_cast<const uint8_t*>(b->user_id) == h0 + L.user;
  if (m->hist_cols > 0)
    packed = packed && b->hist_stride == m->hist_cols &&
             (narrow ? reinterpret_cast<const uint8_t*>(b->hist16)
                     : reinterpret_cast<const uint8_t*>(b->hist)) == h0 + L.hist;
  if (m->dense_feats)
    packed = packed && reinterpret_cast<const uint8_t*>(b->movie_genre) == h0 + L.mg &&
             reinterpret_cast<const uint8_t*>(b->user_genre) == h0 + L.ug &&
             reinterpret_cast<const uint8_t*>(b->numerics) == h0 + L.num;
  if (packed) {
    CUDA_TRY(cudaMemcpyAsync(d, h0, L.total, cudaMemcpyHostToDevice, s.stream));
  } else {
    CUDA_TRY(cudaMemcpyAsync(d + L.movie, b->movie_id, B * 4, cudaMemcpyHostToDevice, s.stream));
    CUDA_TRY(cudaMemcpyAsync(d + L.user, b->user_id, B * 4, cudaMemcpyHostToDevice, s.stream));
    if (m->hist_cols > 0) {
      const size_t es = narrow ? 2 : 4;                       // bytes per history id on the host
      const void* hsrc = narrow ? static_cast<const void*>(b->hist16) : static_cast<const void*>(b->hist);
      if (b->hist_stride == m->hist_cols) {
        CUDA_TRY(cudaMemcpyAsync(d + L.hist, hsrc, B * m->hist_cols * es, cudaMemcpyHostToDevice, s.stream));
      } else {
        CUDA_TRY(cudaMemcpy2DAsync(d + L.hist, (size_t)m->hist_cols * es, hsrc, (size_t)b->hist_stride * es,
                                   (size_t)m->hist_cols * es, B, cudaMemcpyHostToDevice, s.stream));
      }
    }
    if (m->dense_feats) {
      CUDA_TRY(cudaMemcpyAsync(d + L.mg, b->movie_genre, B * 3 * 4, cudaMemcpyHostToDevice, s.stream));
      CUDA_TRY(cudaMemcpyAsync(d + L.ug, b->user_genre, B * 5 * 4, cudaMemcpyHostToDevice, s.stream));
      CUDA_TRY(cudaMemcpyAsync(d + L.num, b->numerics, B * 7 * 4, cudaMemcpyHostToDevice, s.stream));
    }
  }
  BatchView v = packed_view(m, d, L, b->B);
  if (narrow) {
    CUDA_TRY(launch_widen_u16(reinterpret_cast<const uint16_t*>(d + L.hist), s.d_hist32,
                              (int64_t)B * m->hist_cols, s.stream));
    v.hist = s.d_hist32;
  }
  v.probs = probs_out ? probs_out : s.d_probs;
  v.logits = want_logits ? (logits_out ? logits_out : s.d_logits) : nullptr; v.err_flag = slot_err(m, s);
  return launch(m, v, s.stream);
}

// device-visible alias of a host pointer if it is pinned (page-locked) memory, else nullptr
float* pinned_alias(float* p) {
  if (!p) return nullptr;
  cudaPointerAttributes at{};
  if (cudaPointerGetAttributes(&at, p) == cudaSuccess && at.type == cudaMemoryTypeHost && at.devicePointer)
    return static_cast<float*>(at.devicePointer);
  cudaGetLastError();                                   // pageable memory: not an error
  return nullptr;
}

int enqueue_host(srs_model* m, Slot& s, const srs_batch* b, float* probs, float* logits,
                 bool copy_err = true) {
  if (!probs) return fail(SRS_ERR_INVALID, "probs is null");
  // Experimental (SRS_ZERO_COPY_SCORES=1): a pinned output buffer is device-addressable under
  // unified addressing, so the kernel can write the 4 B per row over PCIe itself and the
  // device-to-host copy - one driver call and one copy-engine operation per batch - goes away.
  float* direct = m->zero_copy_scores && b && b->B > 0 ? pinned_alias(probs) : nullptr;   // pageable: the copy
  int rc = stage_and_launch(m, s, b, logits != nullptr, direct);
  if (rc != SRS_OK) return rc;
  if (b->B == 0) return SRS_OK;
  const size_t B = (size_t)b->B;
  if (!direct) CUDA_TRY(cudaMemcpyAsync(probs, s.d_probs, B * 4, cudaMemcpyDeviceToHost, s.stream));
  if (logits) CUDA_TRY(cudaMemcpyAsync(logits, s.d_logits, B * 4, cudaMemcpyDeviceToHost, s.stream));
  if (copy_err)
    CUDA_TRY(cudaMemcpyAsync(s.h_err, slot_err(m, s), sizeof(int), cudaMemcpyDeviceToHost, s.stream));
  return SRS_OK;
}

int wait_slot(srs_model* m, Slot& s) {
  if (!s.stream) return SRS_OK;
  CUDA_TRY(cudaSetDevice(m->device));
  CUDA_TRY(cudaStreamSynchronize(s.stream));
  if (s.h_err && *s.h_err) {
    *s.h_err = 0;
    CUDA_TRY(cudaMemsetAsync(slot_err(m, s), 0, sizeof(int), s.stream));
    CUDA_TRY(cudaStreamSynchronize(s.stream));
    return fail(SRS_ERR_RANGE, "an id in the batch is outside its vocabulary");
  }
  return SRS_OK;
}

int ensure_done(Slot& s, int k) {
  if (!s.h_done) {
    CUDA_TRY(cudaMallocHost(&s.h_done, 4 * sizeof(uint32_t)));
    memset(s.h_done, 0, 4 * sizeof(uint32_t));
  }
  if (k > s.res_capacity) {
    if (s.h_res) cudaFreeHost(s.h_res);
    s.h_res = nullptr; s.res_capacity = 0;
    const int cap = std::max(k, 1024);
    CUDA_TRY(cudaMallocHost(&s.h_res, (size_t)cap * 8));
    s.res_capacity = cap;
  }
  return SRS_OK;
}

// Spin until the call's last kernel has published sequence number `s.seq` (the stream is polled now
// and then so that a failed launch or a faulting kernel ends the wait with an error, not a hang).
int wait_done(srs_model* m, Slot& s) {
  volatile uint32_t* d = s.h_done;
  uint64_t spins = 0;
  while (d[0] != s.seq) {
    if ((++spins & 0x1FFF) == 0) {
      const cudaError_t q = cudaStreamQuery(s.stream);
      if (q == cudaSuccess) {
        if (d[0] == s.seq) break;
        return fail(SRS_ERR_CUDA, "the stream drained without the completion record being written");
      }
      if (q != cudaErrorNotReady) return fail(SRS_ERR_CUDA, "kernel failed: %s", cudaGetErrorString(q));
    }
#if defined(__x86_64__) || defined(__i386__)
    __builtin_ia32_pause();
#endif
  }
  std::atomic_thread_fence(std::memory_order_acquire);
  if (d[1]) return fail(SRS_ERR_RANGE, "an id in the batch is outside its vocabulary");
  (void)m;
  return SRS_OK;
}

// Top k of the n scores in s.d_probs into top_idx / top_scores.  The ranking kernel writes the k positions
// and scores into pinned host memory and then the completion record the caller spins on: no device-to-host
// copy, no stream synchronise.
int rank_scores(srs_model* m, Slot& s, int n, int k, int32_t* top_idx, float* top_scores) {
  int rc = ensure_done(s, k);
  if (rc != SRS_OK) return rc;
  if (k > 0 && n > s.rank_capacity) {
    cudaFree(s.d_rank);
    s.d_rank = nullptr;
    s.rank_capacity = 0;
    const int cap = s.capacity;     // >= n: the scores are in this slot's staging
    CUDA_TRY(cudaMalloc(&s.d_rank, (size_t)cap * 8 + topk_scratch_bytes(cap) + 256));
    s.rank_capacity = cap;
  }
  int32_t* r_idx = s.h_res;
  float* r_top = reinterpret_cast<float*>(s.h_res + s.res_capacity);
  void* scratch = s.d_rank ? s.d_rank + (size_t)s.rank_capacity * 8 : nullptr;
  s.seq += 1;
  CUDA_TRY(launch_topk_done(s.d_probs, n, k, r_idx, r_top, scratch, slot_err(m, s), s.h_done, s.seq, s.stream));
  rc = wait_done(m, s);
  if (k > 0) {
    memcpy(top_idx, r_idx, (size_t)k * 4);
    if (top_scores) memcpy(top_scores, r_top, (size_t)k * 4);
  }
  return rc;
}

}  // namespace

// ======================================================================================
extern "C" {

int srs_abi_version(void) { return SRS_ABI_VERSION; }

const char* srs_last_error(void) { return g_err.c_str(); }

int srs_model_create(const srs_spec* spec, const srs_tensor* tensors, int32_t n_tensors,
                     int32_t device, srs_model** out) {
  if (!spec || !out || (n_tensors > 0 && !tensors)) return fail(SRS_ERR_INVALID, "null argument");
  *out = nullptr;
  if (spec->kind < SRS_EMBEDDINGMLP || spec->kind > SRS_DIEN)
    return fail(SRS_ERR_INVALID, "unknown model kind %d", spec->kind);
  if (spec->emb_dim < 1 || spec->emb_dim > 64) return fail(SRS_ERR_INVALID, "emb_dim must be in 1..64");
  if (spec->n_movies < 1 || spec->n_users < 1 || spec->n_genres < 1)
    return fail(SRS_ERR_INVALID, "vocabulary sizes must be positive");
  if (spec->n_hidden < 0 || spec->n_hidden > 4) return fail(SRS_ERR_INVALID, "n_hidden must be in 0..4");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(SRS_ERR_CUDA, "no CUDA device available (%s); this library has no CPU path",
                cudaGetErrorString(e));
  if (device < 0 || device >= ndev) return fail(SRS_ERR_INVALID, "device %d out of range", device);
  CUDA_TRY(cudaSetDevice(device));
  CUDA_TRY(setup_embmlp_attributes());
  CUDA_TRY(setup_deepfm_attributes());
  CUDA_TRY(setup_din_attributes());
  CUDA_TRY(setup_dien_attributes());
  CUDA_TRY(setup_din_tc_attributes());
  CUDA_TRY(setup_din_rt_attributes());
  CUDA_TRY(setup_din_rt64_attributes());
  CUDA_TRY(setup_embmlp_tc_attributes());
  CUDA_TRY(setup_deepfm_tc_attributes());

  srs_model* m = new srs_model();
  m->spec = *spec;
  m->device = device;
  if (const char* zc = opt("zero_copy_scores", "SRS_ZERO_COPY_SCORES")) {
    m->zero_copy_scores = atoi(zc) == 1;              // pipelined paths too (experimental)
    m->no_zero_copy = atoi(zc) == 0;
  }
  {
    int sms = 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    m->device_sms = sms > 0 ? sms : 148;
  }
  m->EP = round_ep(spec->emb_dim);
  m->hist_cols = (spec->kind == SRS_DIN || spec->kind == SRS_DIEN) ? spec->hist_len
                 : spec->kind == SRS_WIDENDEEP ? 1 : 0;
  m->dense_feats = !(spec->kind == SRS_NEURALCF || spec->kind == SRS_TWOTOWERS);
  m->bytes_per_inf = bytes_per_inference(*spec);
  Builder B{m};
  for (int i = 0; i < n_tensors; ++i)
    if (tensors[i].name) B.by_name[tensors[i].name] = &tensors[i];
  int rc;
  switch (spec->kind) {
    case SRS_NEURALCF:
    case SRS_TWOTOWERS: m->kernel = Kernel::ncf; rc = build_ncf(B); break;
    case SRS_EMBEDDINGMLP:
    case SRS_WIDENDEEP: {
      rc = build_embmlp(B);
      // tensor cores for the reference shape (E <= 12)
      const bool tc = m->EP == 12;
      if (rc == SRS_OK)
        rc = select_kernel(m, "embmlp_impl", "SRS_EMBMLP_IMPL", tc ? Kernel::embmlp_tc : Kernel::embmlp,
                           {{"cudacore", Kernel::embmlp, true, nullptr},
                            {"tc", Kernel::embmlp_tc, tc, "SRS_EMBMLP_IMPL=tc needs emb_dim <= 12"}});
      break;
    }
    case SRS_DEEPFM: {
      rc = build_deepfm(B);
      // tensor-core deep MLP when emb_dim pads to 16
      const bool tc = m->EP == 16;
      if (rc == SRS_OK)
        rc = select_kernel(m, "deepfm_impl", "SRS_DEEPFM_IMPL", tc ? Kernel::deepfm_tc : Kernel::deepfm,
                           {{"cudacore", Kernel::deepfm, true, nullptr},
                            {"tc", Kernel::deepfm_tc, tc, "SRS_DEEPFM_IMPL=tc needs 12 < emb_dim <= 16"}});
      break;
    }
    case SRS_DEEPFM_V2: m->kernel = Kernel::deepfm2; rc = build_deepfm2(B); break;
    case SRS_DIEN: m->kernel = Kernel::dien; rc = build_dien(B); break;
    default: {
      rc = build_din(B);
      // rt: row-tile kernels, E padded to 32 and T in 9..64 (din_rt), E padded to 64 and T in 9..256 (din_rt64);
      // tc: per-pair tensor-core kernel, E padded to 32 and T in 9..128.  Forced, tc and rt also take T <= 8;
      // rtp (the pipelined row-tile kernel, din_rtp.cu) runs only when forced.
      const int T = spec->hist_len;
      const bool tc = m->EP == 32 && T <= 128, rt32 = m->EP == 32 && T <= 64, rt64 = m->EP == 64 && T <= 256;
      const Kernel rt = rt64 ? Kernel::din_rt64 : Kernel::din_rt;
      const Kernel def = T <= 8 ? Kernel::din : (rt32 || rt64) ? rt : tc ? Kernel::din_tc : Kernel::din;
      if (rc == SRS_OK)
        rc = select_kernel(m, "din_impl", "SRS_DIN_IMPL", def,
                           {{"cudacore", Kernel::din, true, nullptr},
                            {"tc", Kernel::din_tc, tc, "SRS_DIN_IMPL=tc needs 16 < emb_dim <= 32 and hist_len <= 128"},
                            {"rtp", Kernel::din_rtp, rt32, "SRS_DIN_IMPL=rtp needs 16 < emb_dim <= 32 and hist_len <= 64"},
                            {"rt", rt, rt32 || rt64,
                             "SRS_DIN_IMPL=rt needs 16 < emb_dim <= 32 and hist_len <= 64, "
                             "or 32 < emb_dim <= 64 and hist_len <= 256"}});
      break;
    }
  }
  // the tensor-core and row-tile kernels read operand images built from the validated reference tensors
  if (rc == SRS_OK) {
    switch (m->kernel) {
      case Kernel::embmlp_tc: rc = build_embmlp_tc(B); break;
      case Kernel::deepfm_tc: rc = build_deepfm_tc(B); break;
      case Kernel::din_tc: rc = build_din_tc(B); break;
      case Kernel::din_rt:
      case Kernel::din_rtp:
      case Kernel::din_rt64: rc = build_din_rt(B); break;
      default: break;
    }
  }
  if (rc == SRS_OK) {
    e = cudaMalloc(&m->err_flag, kErrWords * sizeof(int));
    if (e == cudaSuccess) e = cudaMemset(m->err_flag, 0, kErrWords * sizeof(int));
    if (e != cudaSuccess) rc = fail(SRS_ERR_CUDA, "error-flag allocation failed: %s", cudaGetErrorString(e));
  }
  if (rc == SRS_OK) {
    e = cudaDeviceSynchronize();
    if (e != cudaSuccess) rc = fail(SRS_ERR_CUDA, "weight upload failed: %s", cudaGetErrorString(e));
  }
  if (rc != SRS_OK) {
    std::string keep = g_err;
    srs_model_destroy(m);
    g_err = keep;
    return rc;
  }
  *out = m;
  return SRS_OK;
}

int srs_model_create_ex(const srs_spec* spec, const srs_tensor* tensors, int32_t n_tensors, int32_t device,
                        const char* options, srs_model** out) {
  g_create_opts = options ? options : "";
  const int rc = srs_model_create(spec, tensors, n_tensors, device, out);
  g_create_opts.clear();
  return rc;
}

void srs_model_destroy(srs_model* m) {
  if (!m) return;
  cudaSetDevice(m->device);
  for (Slot& s : m->slots) {
    if (s.stream) { cudaStreamSynchronize(s.stream); cudaStreamDestroy(s.stream); }
    cudaFree(s.d_block); cudaFree(s.d_probs); cudaFree(s.d_logits); cudaFree(s.d_rank);
    cudaFree(s.d_hist32);
    if (s.h_err) cudaFreeHost(s.h_err);
    if (s.h_req) cudaFreeHost(s.h_req);
    if (s.h_done) cudaFreeHost(s.h_done);
    if (s.h_res) cudaFreeHost(s.h_res);
    cudaFree(s.d_req);
  }
  for (void* p : m->owned) cudaFree(p);
  if (m->err_flag) cudaFree(m->err_flag);
  cudaFree(m->movie_feats);
  delete m;
}

int srs_predict_device(srs_model* m, const srs_batch* b, float* probs, float* logits, void* stream) {
  int rc = check_batch(m, b);
  if (rc != SRS_OK) return rc;
  if (!probs) return fail(SRS_ERR_INVALID, "probs is null");
  if (b->B == 0) return SRS_OK;
  BatchView v;
  rc = device_view(m, b, v);
  if (rc != SRS_OK) return rc;
  v.probs = probs; v.logits = logits;
  return launch(m, v, static_cast<cudaStream_t>(stream));
}

// ---- score exchange over peer memory (gather.cu) -------------------------------------------------
int srs_gather_create(int32_t device, int32_t world, int32_t rank, int64_t slice_rows, srs_gather** out) {
  if (!out) return fail(SRS_ERR_INVALID, "null argument");
  PeerGather* g = nullptr;
  cudaError_t e = gather_create(device, world, rank, slice_rows, &g);
  if (e == cudaErrorInvalidValue) return fail(SRS_ERR_INVALID, "need 1 <= world <= 8, 0 <= rank < world, slice_rows >= 1");
  if (e != cudaSuccess) return fail(SRS_ERR_CUDA, "gather buffer allocation failed: %s", cudaGetErrorString(e));
  *out = reinterpret_cast<srs_gather*>(g);
  return SRS_OK;
}

int srs_gather_export(srs_gather* g, void* handle64) {
  if (!g || !handle64) return fail(SRS_ERR_INVALID, "null argument");
  CUDA_TRY(gather_export(reinterpret_cast<PeerGather*>(g), handle64));
  return SRS_OK;
}

int srs_gather_connect(srs_gather* g, const void* handles) {
  if (!g || !handles) return fail(SRS_ERR_INVALID, "null argument");
  CUDA_TRY(gather_connect(reinterpret_cast<PeerGather*>(g), handles));
  return SRS_OK;
}

void srs_gather_destroy(srs_gather* g) { gather_destroy(reinterpret_cast<PeerGather*>(g)); }

int srs_predict_device_gather(srs_model* m, const srs_batch* b, srs_gather* gg, void* stream) {
  int rc = check_batch(m, b);
  if (rc != SRS_OK) return rc;
  PeerGather* g = reinterpret_cast<PeerGather*>(gg);
  if (!g) return fail(SRS_ERR_INVALID, "null gather object");
  if (!gather_connected(g)) return fail(SRS_ERR_INVALID, "srs_gather_connect has not been called");
  if (gather_device(g) != m->device) return fail(SRS_ERR_INVALID, "gather object lives on another device");
  if (b->B < 1 || b->B > gather_slice_rows(g)) return fail(SRS_ERR_INVALID, "batch rows must be in 1..slice_rows");
  BatchView v;
  rc = device_view(m, b, v);
  if (rc != SRS_OK) return rc;
  // kernels ending in gather_signal_tail()
  const bool in_kernel = m->kernel == Kernel::din_rt || m->kernel == Kernel::din_rtp;
  gather_begin_step(g, v, in_kernel);
  rc = launch(m, v, static_cast<cudaStream_t>(stream));
  if (rc != SRS_OK) return rc;
  if (!in_kernel) CUDA_TRY(gather_signal(g, static_cast<cudaStream_t>(stream)));
  return SRS_OK;
}

int srs_gather_wait(srs_gather* g, void* stream) {
  if (!g) return fail(SRS_ERR_INVALID, "null gather object");
  CUDA_TRY(cudaSetDevice(gather_device(reinterpret_cast<PeerGather*>(g))));
  CUDA_TRY(gather_wait(reinterpret_cast<PeerGather*>(g), static_cast<cudaStream_t>(stream)));
  return SRS_OK;
}

int srs_gather_scores(srs_gather* gg, float** scores, int64_t* rows) {
  PeerGather* g = reinterpret_cast<PeerGather*>(gg);
  if (!g || !scores) return fail(SRS_ERR_INVALID, "null argument");
  *scores = gather_buffer(g, gather_parity(g));
  if (rows) *rows = gather_rows(g);
  return SRS_OK;
}

int srs_gather_copy_scores(srs_gather* gg, float* dst, int32_t dst_on_host, void* stream) {
  PeerGather* g = reinterpret_cast<PeerGather*>(gg);
  if (!g || !dst) return fail(SRS_ERR_INVALID, "null argument");
  CUDA_TRY(cudaSetDevice(gather_device(g)));
  CUDA_TRY(cudaMemcpyAsync(dst, gather_buffer(g, gather_parity(g)), (size_t)gather_rows(g) * 4,
                           dst_on_host ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice,
                           static_cast<cudaStream_t>(stream)));
  return SRS_OK;
}

int srs_predict_host(srs_model* m, const srs_batch* b, float* probs, float* logits) {
  if (!m) return fail(SRS_ERR_INVALID, "null model");
  std::lock_guard<std::mutex> lock(m->mu);
  Slot& s = m->slots[kSlots];
  // Latency path: when the caller's output buffers are pinned, the kernel writes the scores (4 B per row)
  // straight into them over PCIe and a one-warp kernel publishes the completion record: two copy-engine
  // operations, two driver calls and the stream synchronise of the general path go away.
  if (probs && b && b->B > 0 && !m->no_zero_copy) {
    float* dp = pinned_alias(probs);
    float* dl = logits ? pinned_alias(logits) : nullptr;
    if (dp && (!logits || dl)) {
      int rc = ensure_slot(m, s, b->B);
      if (rc == SRS_OK) rc = ensure_done(s, 0);
      if (rc != SRS_OK) return rc;
      rc = stage_and_launch(m, s, b, logits != nullptr, dp, dl);
      if (rc != SRS_OK) return rc;
      s.seq += 1;
      CUDA_TRY(launch_finish(slot_err(m, s), s.h_done, s.seq, s.stream));
      return wait_done(m, s);
    }
  }
  int rc = enqueue_host(m, s, b, probs, logits);
  if (rc != SRS_OK) return rc;
  return wait_slot(m, s);
}

int srs_predict_host_batches(srs_model* m, int32_t n, const srs_batch* batches,
                             float* const* probs, float* const* logits) {
  if (!m) return fail(SRS_ERR_INVALID, "null model");
  if (n < 0 || (n > 0 && (!batches || !probs))) return fail(SRS_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> lock(m->mu);
  CUDA_TRY(cudaSetDevice(m->device));
  int rc = SRS_OK;
  for (int i = 0; i < n && rc == SRS_OK; ++i) {
    Slot& s = m->slots[i % kSlots];
    if (i >= kSlots) CUDA_TRY(cudaStreamSynchronize(s.stream));     // slot's previous batch is out
    rc = enqueue_host(m, s, &batches[i], probs[i], logits ? logits[i] : nullptr, false);
  }
  for (int k = 0; k < kSlots; ++k)
    if (m->slots[k].stream) {
      cudaError_t e = cudaStreamSynchronize(m->slots[k].stream);
      if (e != cudaSuccess && rc == SRS_OK)
        rc = fail(SRS_ERR_CUDA, "stream synchronize failed: %s", cudaGetErrorString(e));
    }
  if (rc != SRS_OK) return rc;
  int flags[kSlots] = {0};
  CUDA_TRY(cudaMemcpy(flags, m->err_flag + 1, kSlots * sizeof(int), cudaMemcpyDeviceToHost));
  bool any = false;
  for (int k = 0; k < kSlots; ++k) any = any || flags[k] != 0;
  if (any) {
    CUDA_TRY(cudaMemset(m->err_flag + 1, 0, kSlots * sizeof(int)));
    return fail(SRS_ERR_RANGE, "an id in a batch was outside its vocabulary");
  }
  return SRS_OK;
}

int srs_num_slots(void) { return kSlots; }

int srs_predict_host_async(srs_model* m, int32_t slot, const srs_batch* b, float* probs,
                           float* logits) {
  if (!m) return fail(SRS_ERR_INVALID, "null model");
  if (slot < 0 || slot >= kSlots) return fail(SRS_ERR_INVALID, "slot %d out of range", slot);
  return enqueue_host(m, m->slots[slot], b, probs, logits);
}

int srs_wait_slot(srs_model* m, int32_t slot) {
  if (!m) return fail(SRS_ERR_INVALID, "null model");
  if (slot < 0 || slot >= kSlots) return fail(SRS_ERR_INVALID, "slot %d out of range", slot);
  return wait_slot(m, m->slots[slot]);
}

int srs_model_status(srs_model* m) {
  if (!m) return fail(SRS_ERR_INVALID, "null model");
  CUDA_TRY(cudaSetDevice(m->device));
  CUDA_TRY(cudaDeviceSynchronize());
  if (m->kernel == Kernel::din_rtp) {                // a protocol error in din_rtp_kernel ends the launch, see rtp_wait
    int aborted = 0;
    unsigned long long rec[4] = {0, 0, 0, 0};
    CUDA_TRY(take_din_rtp_abort(&aborted, rec));
    if (aborted)
      return fail(SRS_ERR_CUDA, "din_rtp_kernel: an mbarrier wait timed out (wait code %llu, block %llu, thread %llu, "
                  "parity %llu); the scores of that launch are invalid", rec[0], rec[1], rec[2], rec[3]);
  }
  if (m->kernel == Kernel::din_rt64) {               // -DRT64_WATCHDOG builds of din_rt64.cu only
    int n = 0;
    unsigned long long rec[64];
    CUDA_TRY(take_din_rt64_abort(&n, rec));
    if (n > 0) {
      char msg[900];
      int at = snprintf(msg, sizeof(msg), "din_rt64_kernel: %d mbarrier wait(s) timed out [line/block/thread/parity]:", n);
      for (int i = 0; i < n && at < (int)sizeof(msg) - 60; ++i)
        at += snprintf(msg + at, sizeof(msg) - at, " %llu/%llu/%llu/%llu", rec[4 * i], rec[4 * i + 1],
                       rec[4 * i + 2] & 0xffffffffull, rec[4 * i + 3]);
      return fail(SRS_ERR_CUDA, "%s", msg);
    }
  }
  int flags[kErrWords] = {0};
  CUDA_TRY(cudaMemcpy(flags, m->err_flag, kErrWords * sizeof(int), cudaMemcpyDeviceToHost));
  bool any = false;
  for (int k = 0; k < kErrWords; ++k) any = any || flags[k] != 0;
  if (any) {
    CUDA_TRY(cudaMemset(m->err_flag, 0, kErrWords * sizeof(int)));
    return fail(SRS_ERR_RANGE, "an id in a batch was outside its vocabulary");
  }
  return SRS_OK;
}

int64_t srs_model_bytes_per_inference(const srs_model* m) { return m ? m->bytes_per_inf : 0; }

const char* srs_model_kernel_name(const srs_model* m) { return m ? kernel_name(m) : ""; }

int srs_model_set_sm_limit(srs_model* m, int32_t n_sms) {
  if (!m) return fail(SRS_ERR_INVALID, "null model");
  const int n = (n_sms <= 0 || n_sms > m->device_sms) ? m->device_sms : n_sms;
  std::lock_guard<std::mutex> lock(m->mu);
  switch (m->kernel) {
    case Kernel::din_rt:
    case Kernel::din_rtp:
    case Kernel::din_rt64: m->din_rt.num_sms = n; break;
    case Kernel::din_tc: m->din_tc.num_sms = n; break;
    case Kernel::embmlp_tc: m->emb_tc.num_sms = n; break;
    case Kernel::deepfm_tc: m->fm_tc.num_sms = n; break;
    default: break;                                  // the CUDA-core kernels take no SM limit
  }
  return SRS_OK;
}

int64_t srs_launch_count(void) { return g_launch_count; }

int srs_fill_uniform(float* device_ptr, int64_t n, uint64_t seed, float lo, float hi,
                     int32_t device, void* stream) {
  if (!device_ptr && n > 0) return fail(SRS_ERR_INVALID, "null pointer");
  CUDA_TRY(cudaSetDevice(device));
  CUDA_TRY(launch_fill_uniform(device_ptr, n, seed, lo, hi, static_cast<cudaStream_t>(stream)));
  return SRS_OK;
}

int srs_cosine_scores_device(const float* query, const float* cands, int32_t n, int32_t dim,
                             float* scores, int32_t device, void* stream) {
  if ((!query || !cands || !scores) && n > 0) return fail(SRS_ERR_INVALID, "null pointer");
  if (dim < 1) return fail(SRS_ERR_INVALID, "dim must be positive");
  CUDA_TRY(cudaSetDevice(device));
  CUDA_TRY(launch_cosine(query, cands, n, dim, scores, static_cast<cudaStream_t>(stream)));
  return SRS_OK;
}

int srs_topk_device(const float* scores, int32_t n, int32_t k, int32_t* top_idx,
                    float* top_scores, int32_t device, void* stream) {
  if (n < 0 || k < 0) return fail(SRS_ERR_INVALID, "negative n or k");
  if (n == 0 || k == 0) return SRS_OK;
  if (!scores || !top_idx) return fail(SRS_ERR_INVALID, "null pointer");
  if (n > (1 << 30)) return fail(SRS_ERR_INVALID, "at most 2^30 scores");
  CUDA_TRY(cudaSetDevice(device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  void* scratch = nullptr;
  const size_t need = topk_scratch_bytes(n);
  if (need) CUDA_TRY(cudaMallocAsync(&scratch, need, s));
  cudaError_t e = launch_topk(scores, n, k, top_idx, top_scores, scratch, s);
  if (scratch) cudaFreeAsync(scratch, s);
  CUDA_TRY(e);
  return SRS_OK;
}

int srs_rank_host(srs_model* m, const srs_batch* b, int32_t k, int32_t* top_idx,
                  float* top_scores) {
  if (!m) return fail(SRS_ERR_INVALID, "null model");
  if (k < 0) return fail(SRS_ERR_INVALID, "negative k");
  std::lock_guard<std::mutex> lock(m->mu);
  Slot& s = m->slots[kSlots];
  int rc = stage_and_launch(m, s, b, false);
  if (rc != SRS_OK) return rc;
  const int n = b->B;
  if (n == 0) return SRS_OK;
  if (k > n) k = n;
  if (k > 0 && !top_idx) return fail(SRS_ERR_INVALID, "top_idx is null");
  return rank_scores(m, s, n, k, top_idx, top_scores);
}

int srs_model_set_movie_features(srs_model* m, int32_t n_movies, const int32_t* genres, const float* numerics) {
  if (!m) return fail(SRS_ERR_INVALID, "null model");
  if (n_movies < 1 || !genres || !numerics) return fail(SRS_ERR_INVALID, "null or empty movie feature table");
  std::lock_guard<std::mutex> lock(m->mu);
  CUDA_TRY(cudaSetDevice(m->device));
  std::vector<int32_t> packed((size_t)n_movies * 8, 0);
  for (int i = 0; i < n_movies; ++i) {
    for (int g = 0; g < 3; ++g) {
      const int32_t v = genres[(size_t)i * 3 + g];
      if (v >= m->spec.n_genres) return fail(SRS_ERR_RANGE, "movie %d: genre index %d outside the vocabulary", i, v);
      packed[(size_t)i * 8 + g] = v < 0 ? -1 : v;
    }
    memcpy(&packed[(size_t)i * 8 + 3], numerics + (size_t)i * 4, 16);
  }
  cudaFree(m->movie_feats);
  m->movie_feats = nullptr; m->movie_feats_rows = 0;
  CUDA_TRY(cudaMalloc(&m->movie_feats, packed.size() * 4));
  CUDA_TRY(cudaMemcpy(m->movie_feats, packed.data(), packed.size() * 4, cudaMemcpyHostToDevice));
  m->movie_feats_rows = n_movies;
  return SRS_OK;
}

int srs_rank_user_host(srs_model* m, const srs_user_row* user, const int32_t* cand, int32_t n, int32_t k,
                       int32_t* top_idx, float* top_scores, float* probs) {
  if (!m) return fail(SRS_ERR_INVALID, "null model");
  if (!user || (n > 0 && !cand) || n < 0 || k < 0) return fail(SRS_ERR_INVALID, "bad argument");
  if (m->dense_feats && !m->movie_feats)
    return fail(SRS_ERR_INVALID, "this model reads movie features: call srs_model_set_movie_features first");
  const int hc = m->hist_cols;
  if (user->n_hist < 0 || user->n_hist > hc || (user->n_hist > 0 && !user->hist))
    return fail(SRS_ERR_INVALID, "n_hist must be in 0..%d", hc);
  std::lock_guard<std::mutex> lock(m->mu);
  Slot& s = m->slots[kSlots];
  CUDA_TRY(cudaSetDevice(m->device));
  int rc = ensure_slot(m, s, n);
  if (rc != SRS_OK) return rc;
  if (n == 0) return SRS_OK;
  if (k > n) k = n;
  if (k > 0 && !top_idx) return fail(SRS_ERR_INVALID, "top_idx is null");
  if (n > s.req_capacity || !s.d_req) {
    cudaFree(s.d_req);
    if (s.h_req) cudaFreeHost(s.h_req);
    s.d_req = nullptr; s.h_req = nullptr; s.req_capacity = 0;
    const size_t words = 16 + (size_t)hc + (size_t)s.capacity;
    CUDA_TRY(cudaMalloc(&s.d_req, words * 4));
    CUDA_TRY(cudaMallocHost(&s.h_req, words * 4));
    s.req_capacity = s.capacity;
  }
  // request block: [userId | userGenre1..5 | 3 user numerics | hist[hc] | candidate ids[n]]
  int32_t* h = s.h_req;
  h[0] = user->user_id;
  for (int g = 0; g < 5; ++g) h[1 + g] = user->user_genre[g] < 0 ? -1 : user->user_genre[g];
  memcpy(h + 6, user->user_numerics, 12);
  for (int t = 0; t < hc; ++t) h[9 + t] = t < user->n_hist ? user->hist[t] : 0;     // 0 = the padding id
  memcpy(h + 9 + hc, cand, (size_t)n * 4);
  // one small copy: (9 + T + n) words instead of n full feature rows.  (Letting the assemble kernel read the
  // pinned block over PCIe itself was measured slower: every row re-reads the user part from host memory.)
  CUDA_TRY(cudaMemcpyAsync(s.d_req, s.h_req, (9 + (size_t)hc + (size_t)n) * 4, cudaMemcpyHostToDevice, s.stream));
  const PackedLayout L = packed_layout(m, (size_t)n);
  uint8_t* d = s.d_block;
  BatchView v = packed_view(m, d, L, n);
  v.probs = s.d_probs; v.logits = nullptr; v.err_flag = slot_err(m, s);
  CUDA_TRY(launch_assemble_request(s.d_req, m->movie_feats, m->movie_feats_rows, n, hc, m->dense_feats ? 1 : 0,
                                   reinterpret_cast<int32_t*>(d + L.movie), reinterpret_cast<int32_t*>(d + L.user),
                                   reinterpret_cast<int32_t*>(d + L.hist), reinterpret_cast<int32_t*>(d + L.mg),
                                   reinterpret_cast<int32_t*>(d + L.ug), reinterpret_cast<float*>(d + L.num),
                                   slot_err(m, s), s.stream));
  rc = launch(m, v, s.stream);
  if (rc != SRS_OK) return rc;
  if (probs) CUDA_TRY(cudaMemcpyAsync(probs, s.d_probs, (size_t)n * 4, cudaMemcpyDeviceToHost, s.stream));
  return rank_scores(m, s, n, k, top_idx, top_scores);
}

int srs_debug_din_trace(srs_model* m, int32_t enable, uint64_t* out40) {
  if (!m) return fail(SRS_ERR_INVALID, "null model");
  CUDA_TRY(cudaSetDevice(m->device));
  m->din_tc.trace = enable;
  m->din_rt.trace = enable;
  if (out40) {
    CUDA_TRY(cudaDeviceSynchronize());
    unsigned long long* out = reinterpret_cast<unsigned long long*>(out40);
    switch (m->kernel) {
      case Kernel::din_rtp: CUDA_TRY(read_din_rtp_trace(out)); break;
      case Kernel::din_rt: CUDA_TRY(read_din_rt_trace(out)); break;
      default: CUDA_TRY(read_din_tc_trace(out)); break;
    }
  }
  return SRS_OK;
}

int srs_debug_din_timeline(srs_model* m, uint64_t* out512) {   /* 12 x 64 values */
  if (!m || !out512) return fail(SRS_ERR_INVALID, "null argument");
  if (m->kernel != Kernel::din_rtp) return fail(SRS_ERR_INVALID, "the per-tile timeline exists for din_rtp_kernel only");
  CUDA_TRY(cudaSetDevice(m->device));
  CUDA_TRY(cudaDeviceSynchronize());
  CUDA_TRY(read_din_rtp_timeline(reinterpret_cast<unsigned long long*>(out512)));
  return SRS_OK;
}

int srs_debug_umma_bench(int32_t N, int32_t n_mma, int32_t a_in_tmem, int32_t two_acc,
                         int32_t device, uint64_t* out2) {
  if (!out2 || (N != 32 && N != 64 && N != 128) || n_mma < 1 || n_mma > 4096)
    return fail(SRS_ERR_INVALID, "bad argument");
  CUDA_TRY(cudaSetDevice(device));
  unsigned long long* d = nullptr;
  CUDA_TRY(cudaMalloc(&d, 16));
  cudaError_t e = launch_umma_bench(d, N, n_mma, a_in_tmem & 1, two_acc & 1, (two_acc >> 1) & 1, nullptr);
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e == cudaSuccess) e = cudaMemcpy(out2, d, 16, cudaMemcpyDeviceToHost);
  cudaFree(d);
  if (e != cudaSuccess) return fail(SRS_ERR_CUDA, "umma bench failed: %s", cudaGetErrorString(e));
  return SRS_OK;
}

int srs_selftest_umma(const float* A, const float* B, float* D, int32_t N, int32_t k_blocks,
                      int32_t a_in_tmem, int32_t device) {
  if (!A || !B || !D) return fail(SRS_ERR_INVALID, "null pointer");
  CUDA_TRY(cudaSetDevice(device));
  CUDA_TRY(launch_umma_selftest(A, B, D, N, k_blocks, a_in_tmem, nullptr));
  CUDA_TRY(cudaDeviceSynchronize());
  return SRS_OK;
}

}  // extern "C"
