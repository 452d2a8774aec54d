/*
 * srs_ctr.h - C ABI of the B200-native SparrowRecSys CTR ranking forward path.
 *
 * The reference has no FFI: its hot path is `model.predict(feature_dict)` on a
 * Keras graph (TFRecModel/src/com/sparrowrecsys/offline/tensorflow/<Model>.py) and, at
 * serve time, the same graph behind TF-Serving's REST `:predict`
 * (src/main/java/com/sparrowrecsys/online/recprocess/RecForYouProcess.java:113-138).
 * This header is the boundary a maintainer binds instead (ctypes stub in
 * sparrowrecsys_b200/_lib.py, JNI sketch in INTEGRATION.md).  Each entry point
 * cites the reference interface it replaces.
 *
 * Conventions: plain pointers and sizes only; every function returns SRS_OK (0)
 * or a negative error code and never throws across the ABI; srs_last_error()
 * gives the message of the last failure on the calling thread.  The caller owns
 * all input/output buffers; the library owns its device copy of the weights.
 */
#ifndef SRS_CTR_H_
#define SRS_CTR_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SRS_ABI_VERSION 3

enum srs_status {
  SRS_OK = 0,
  SRS_ERR_INVALID = -1,     /* bad argument / unsupported spec                   */
  SRS_ERR_MISSING = -2,     /* a required weight tensor was not supplied         */
  SRS_ERR_SHAPE = -3,       /* a weight tensor has the wrong shape               */
  SRS_ERR_CUDA = -4,        /* CUDA runtime failure (message has the cudaError)  */
  SRS_ERR_RANGE = -5,       /* an id in the batch is outside its vocabulary:     */
                            /* mirrors TF's assert_less_than_num_buckets         */
  SRS_ERR_NOMEM = -6
};

/* Model families = the reference's model scripts. */
enum srs_model_kind {
  SRS_EMBEDDINGMLP = 0,     /* EmbeddingMLP.py:72-77                             */
  SRS_WIDENDEEP = 1,        /* WideNDeep.py:101-108                              */
  SRS_NEURALCF = 2,         /* NeuralCF.py:45-53  (neural_cf_model_1)            */
  SRS_TWOTOWERS = 3,        /* NeuralCF.py:57-70  (neural_cf_model_2)            */
  SRS_DEEPFM = 4,           /* DeepFM.py:91-113                                  */
  SRS_DEEPFM_V2 = 5,        /* DeepFM_v2.py:98-155                               */
  SRS_DIN = 6,              /* DIN.py:125-167                                    */
  SRS_DIEN = 7              /* DIEN.py:154-256 (y_pred; AUGRU initial state is the  */
                            /* stored tensor "augru_h0", emb_dim <= 32)            */
};

/* Hyper-parameters the reference hard-codes as module constants
 * (DIN.py:30-31,66,132; EmbeddingMLP.py:50-58; NeuralCF.py:74). */
typedef struct srs_spec {
  int32_t kind;             /* enum srs_model_kind                               */
  int32_t emb_dim;          /* E                                                 */
  int32_t n_movies;         /* num_buckets of movieId (valid ids 0..n-1)         */
  int32_t n_users;          /* num_buckets of userId                             */
  int32_t n_genres;         /* 19                                                */
  int32_t hist_len;         /* T (DIN, DIEN); W&D reads history slot 0 only      */
  int32_t n_hidden;         /* entries used in hidden[]                          */
  int32_t hidden[4];        /* MLP widths, model dependent                       */
  int32_t au_hidden;        /* DIN activation-unit / DIEN attention width (32)   */
  int32_t cross_buckets;    /* W&D hash_bucket_size (10000)                      */
  int32_t proj_dim;         /* DeepFM_v2 field projection width (64)             */
  int32_t final_dense;      /* two towers: Dense(1,sigmoid) after the dot        */
} srs_spec;

enum srs_location { SRS_HOST = 0, SRS_DEVICE_BORROWED = 1 };

/* One weight tensor in the reference's own (Keras variable) shape: Dense kernels
 * [in,out], tables [buckets,E], vectors [n] as rows=n, cols=1.  Names are the
 * canonical ones of sparrowrecsys_b200/weights.py (SURVEY.md appendix A).
 * SRS_DEVICE_BORROWED: `data` is a device pointer on the model's device that the
 * library uses in place (no copy; must outlive the model; only for embedding
 * tables whose emb_dim is a multiple of 4) - this is how a 25.6 GB table is
 * handed over without a host round trip. */
typedef struct srs_tensor {
  const char* name;
  const float* data;
  int64_t rows;
  int64_t cols;
  int32_t location;         /* enum srs_location                                 */
} srs_tensor;

/* One batch of ranking instances, structure-of-arrays.  Replaces the feature
 * dict handed to `model.predict` (keys of the Keras `inputs` dicts, e.g.
 * DIN.py:34-59) / the `instances` array of the TF-Serving request
 * (RecForYouProcess.java:118-127).  Genre strings are already vocabulary indices
 * (-1 = missing / out of vocabulary -> zero vector), integer numerics already
 * cast to float32 (what numeric_column does).  Pointers a model does not read may
 * be NULL.  All pointers are host pointers for srs_predict_host* and device
 * pointers (on the model's device) for srs_predict_device.
 * Fast path for host batches: when the arrays lie back to back in memory in the order
 * movie_id, user_id, hist (hist_stride == T), movie_genre, user_genre, numerics (arrays the
 * model does not read left out), srs_predict_host* moves the whole batch with ONE
 * host-to-device copy instead of one per array. */
typedef struct srs_batch {
  int32_t B;                   /* rows                                            */
  int32_t hist_stride;         /* elements between consecutive rows of `hist`     */
  const int32_t* movie_id;     /* [B]                                             */
  const int32_t* user_id;      /* [B]                                             */
  const int32_t* hist;         /* [B, T] userRatedMovie<k> in graph position order */
  const int32_t* movie_genre;  /* [B, 3] movieGenre1..3                           */
  const int32_t* user_genre;   /* [B, 5] userGenre1..5                            */
  const float* numerics;       /* [B, 7] movieAvgRating, movieRatingCount,
                                  movieRatingStddev, releaseYear, userAvgRating,
                                  userRatingCount, userRatingStddev               */
  const uint16_t* hist16;      /* host batches only, optional: the history ids as uint16
                                  [B, T] (same stride and order as `hist`, which is then
                                  ignored) for vocabularies of at most 65536 movies - the
                                  history is most of a DIN batch, so this halves the bytes
                                  that cross PCIe; widened to int32 on the device.  In the
                                  packed layout it takes the place of `hist`, padded to a
                                  multiple of 4 bytes.  NULL otherwise.                 */
} srs_batch;

typedef struct srs_model srs_model;

int srs_abi_version(void);

/* Message of the last error raised on this thread ("" if none). */
const char* srs_last_error(void);

/* Build a model on CUDA device `device`: validates names/shapes against `spec`,
 * copies (and privately re-lays-out) the weights into HBM.  Replaces building
 * the module-level Keras `model` and loading its variables (e.g. DIN.py:169,
 * NeuralCF.py:74 + the SavedModel under webroot/modeldata/). */
int srs_model_create(const srs_spec* spec, const srs_tensor* tensors, int32_t n_tensors,
                     int32_t device, srs_model** out);

/* Same, with kernel-variant options "key=value;key=value": din_impl = rt | rtp | tc | cudacore,
 * embmlp_impl / deepfm_impl = tc | cudacore, zero_copy_scores = 0 | 1.  Unknown keys are ignored; a
 * forced variant that does not support the shape makes the call fail.  NULL / "" = the defaults
 * (which srs_model_kernel_name reports).  The environment variables SRS_DIN_IMPL, SRS_EMBMLP_IMPL,
 * SRS_DEEPFM_IMPL, SRS_ZERO_COPY_SCORES are read only for keys the string does not set. */
int srs_model_create_ex(const srs_spec* spec, const srs_tensor* tensors, int32_t n_tensors,
                        int32_t device, const char* options, srs_model** out);

void srs_model_destroy(srs_model* m);

/* Forward pass with everything resident in HBM; asynchronous on `stream`
 * (a cudaStream_t; NULL = the default stream).  `probs` [B] receives the model
 * output (sigmoid probability; raw dot for two towers without final dense);
 * `logits` [B] (may be NULL) receives the pre-sigmoid value.  Replaces the
 * compiled forward that `model.predict` runs per batch (e.g. DIN.py:185).
 * Out-of-range ids are read as id 0 and latch an error flag that
 * srs_model_status() reports. */
int srs_predict_device(srs_model* m, const srs_batch* batch, float* probs, float* logits,
                       void* stream);

/* ---- One ranking call that spans the GPUs of a box (RecForYouProcess.java:56-59,92-94 with the
 * candidate list sharded by rows, SURVEY.md section 8e): every rank needs every rank's scores.
 * Instead of kernel + all-gather, each rank's forward kernel stores its scores into its slice of
 * EVERY rank's gather buffer over NVLink (CUDA IPC peer mappings), followed by one flag word per
 * rank.  One process per GPU; `slice_rows` = rows per rank (the last rank may score fewer).
 *   1. every rank: srs_gather_create, srs_gather_export -> 64-byte handle
 *   2. exchange the handles (torch.distributed / MPI / a pipe), every rank: srs_gather_connect with
 *      the world x 64 bytes in rank order
 *   3. per call: srs_predict_device_gather (asynchronous on `stream`), then srs_gather_wait on the
 *      stream that consumes the scores, then srs_gather_scores for the device pointer of the full
 *      [world * slice_rows] vector (valid until the call after the next one: two buffers alternate).
 * Every rank must make the same sequence of calls.  The step counters live on the device, so a
 * sequence of an EVEN number of predict / wait pairs can be captured in a CUDA graph and replayed
 * (the buffer parity of each pair is fixed at capture). */
typedef struct srs_gather srs_gather;
int srs_gather_create(int32_t device, int32_t world, int32_t rank, int64_t slice_rows, srs_gather** out);
int srs_gather_export(srs_gather* g, void* handle64);
int srs_gather_connect(srs_gather* g, const void* handles /* world * 64 bytes, rank order */);
void srs_gather_destroy(srs_gather* g);
int srs_predict_device_gather(srs_model* m, const srs_batch* batch, srs_gather* g, void* stream);
int srs_gather_wait(srs_gather* g, void* stream);
int srs_gather_scores(srs_gather* g, float** scores, int64_t* rows);
/* copy the gathered vector of the latest call to `dst` (device or host memory), asynchronous on `stream` */
int srs_gather_copy_scores(srs_gather* g, float* dst, int32_t dst_on_host, void* stream);

/* Forward pass from host buffers: H2D of the batch, kernel, D2H of the scores,
 * synchronous.  This is the drop-in for `model.predict(dict) -> float32[B,1]`
 * and for one TF-Serving `:predict` call.  Returns SRS_ERR_RANGE if an id was
 * out of range (outputs are still written). */
int srs_predict_host(srs_model* m, const srs_batch* batch, float* probs, float* logits);

/* A whole dataset in batches, the way `model.predict(dataset)` iterates it (e.g.
 * DIN.py:185 over make_csv_dataset batches): batch i is copied in, scored and copied out
 * on internal slot i % srs_num_slots(), so the PCIe copies of one batch overlap the kernel
 * of another.  Synchronous; probs[i] (and logits[i] if `logits` != NULL) receive batch i.
 * Host buffers should be pinned for the copies to overlap.  Not to be mixed concurrently
 * with srs_predict_host_async on the same model. */
int srs_predict_host_batches(srs_model* m, int32_t n_batches, const srs_batch* batches,
                             float* const* probs, float* const* logits);

/* Pipelined variant: enqueue on one of srs_num_slots() internal slots (each with
 * its own stream and device staging) and return; srs_wait_slot() blocks until that
 * slot's scores are in `probs`.  Host buffers must stay valid (and should be
 * pinned for the copies to overlap) until the wait returns. */
int srs_num_slots(void);
int srs_predict_host_async(srs_model* m, int32_t slot, const srs_batch* batch, float* probs,
                           float* logits);
int srs_wait_slot(srs_model* m, int32_t slot);

/* Synchronises the device and reports SRS_ERR_RANGE if any kernel since the last
 * call saw an out-of-range id, SRS_ERR_CUDA on a sticky CUDA error. */
int srs_model_status(srs_model* m);

/* Algorithmic bytes per inference of this model (SURVEY.md section 8d definition). */
int64_t srs_model_bytes_per_inference(const srs_model* m);

/* Name of the kernel variant srs_predict_* dispatches to for this model.  DIN has four
 * (din_rt_kernel / din_rt64_kernel: tcgen05 row tiles; din_tc_kernel: tcgen05 per pair;
 * din_kernel: CUDA cores); the choice follows the shape and can be forced with the environment
 * variable SRS_DIN_IMPL = rt | rtp | tc | cudacore read by srs_model_create (a forced variant that does
 * not support the shape makes srs_model_create fail; rtp selects din_rtp_kernel, the row-tile kernel with
 * the phases of consecutive row groups pipelined, see csrc/din_rtp.cu).  SRS_EMBMLP_IMPL and SRS_DEEPFM_IMPL
 * (tc | cudacore) do the same for EmbeddingMLP / Wide&Deep and DeepFM. */
const char* srs_model_kernel_name(const srs_model* m);

/* Limit the persistent tensor-core kernels of this model (din_rt / din_rt64 / din_tc /
 * embmlp_tc / deepfm_tc) to at most n_sms CTAs per launch (n_sms <= 0: every SM of the device,
 * the default).  A launch then leaves the other SMs to launches of other streams: with
 * 148 / S CTAs per launch, S consecutive batches of a pipeline run side by side on disjoint SM
 * sets, each CTA walking several row groups, so the per-launch latency chain (prologue, first
 * ids, launch gap) is paid once per S batches per SM instead of once per batch.  Takes effect
 * at the next srs_predict_* call; results do not depend on it. */
int srs_model_set_sm_limit(srs_model* m, int32_t n_sms);

/* Number of kernels this library has launched in this process (all models). */
int64_t srs_launch_count(void);

/* Deterministic counter-based fill of a device float buffer:
 * x[i] = lo + (hi-lo) * u(seed, i), u in [0,1) from a splitmix64 hash of (seed, i).
 * Used to initialise synthetic embedding tables in place (BASELINE cfg 5). */
int srs_fill_uniform(float* device_ptr, int64_t n, uint64_t seed, float lo, float hi,
                     int32_t device, void* stream);

/* Batched cosine similarity of one query embedding against n candidates
 * (online/model/Embedding.java:33-47, used by SimilarMovieProcess.java:121-137
 * and RecForYouProcess.java:93-105).  Device pointers. */
int srs_cosine_scores_device(const float* query, const float* cands, int32_t n, int32_t dim,
                             float* scores, int32_t device, void* stream);

/* Ranking tail of both online rankers: order n candidate scores descending and return the
 * first min(k, n) positions (and, if top_scores != NULL, their scores).  Replaces
 * `candidateScoreMap.entrySet().stream().sorted(comparingByValue(reverseOrder()))` +
 * `subList(0, size)` (RecForYouProcess.java:56-59,92-94; SimilarMovieProcess.java:26-31,
 * 133-135).  Order of Double.compareTo: NaN ranks first, -0.0 after 0.0; equal scores - in
 * HashMap iteration order in the reference, i.e. unspecified - rank by position, lower
 * first.  Device pointers; asynchronous on `stream`. */
int srs_topk_device(const float* scores, int32_t n, int32_t k, int32_t* top_idx,
                    float* top_scores, int32_t device, void* stream);

/* ---- Candidate retrieval: exact top-k over an item index resident in HBM.  Replaces the recall stage
 * in front of the rankers: SimilarMovieProcess.retrievalCandidatesByEmbedding (SimilarMovieProcess.java:91-112,
 * which scores the whole catalog by Embedding.calculateSimilarity) and the fixed candidate list of
 * RecForYouProcess.getRecList (RecForYouProcess.java:34-35, getMovies(800, "rating")); the output feeds
 * srs_rank_user_host.  Unlike SimilarMovieProcess.java:104 (an ascending sort, which keeps the LEAST similar
 * movies) the result is the most similar first, as the ranker (SimilarMovieProcess.java:135) intends.
 *
 * srs_index_create: an index over n items [n][dim] float32 (1 <= n < 2^31, 1 <= dim <= 128).  The library
 * keeps a bf16 scan copy (cosine: of the unit-length rows), per-row norms, and the float32 rows for exact
 * rescoring: copied from host memory (SRS_HOST), or used in place when `items` is a device pointer on
 * `device` (SRS_DEVICE_BORROWED; it must outlive the index).
 * Scores: SRS_DOT = float32 fmaf chain over k = 0..dim-1; SRS_COSINE = Embedding.calculateSimilarity
 * (online/model/Embedding.java:33-47), bit for bit what srs_cosine_scores_device gives for the pair.  A zero
 * row's cosine is 0/0 = NaN and, as in the reference's Double ordering, ranks first. */
enum srs_metric { SRS_DOT = 0, SRS_COSINE = 1 };
typedef struct srs_index srs_index;
int srs_index_create(const float* items, int64_t n, int32_t dim, int32_t metric, int32_t location,
                     int32_t device, srs_index** out);
void srs_index_destroy(srs_index* index);

/* Search q queries [q][dim] (dim must equal the index's), 1 <= k <= 1024, `exclude` [q] an item position
 * per query to leave out (-1 = none; NULL = none for every query).  For each query: top_pos [q][k] and
 * top_scores [q][k] receive the best min(k, eligible) positions, best first, in the order of
 * srs_topk_device (descending score, NaN first, -0.0 after 0.0, equal scores by lower position), and their
 * exact scores; unused slots get position -1 and score 0.  No q x n score matrix is formed and the result
 * does not depend on timing.
 * srs_index_search_device: device pointers, queued on `stream`; it synchronises `stream` once per block of
 * 256 queries, and again for each extra pass a query whose candidates overflow needs.  Calls on one index
 * are serialised, also across streams: a search waits on the device for the previous search of the same
 * index to finish (its working lists are per index).
 * srs_index_search_host: host pointers, synchronous.
 * An exclude position outside -1..n-1 is SRS_ERR_INVALID. */
int srs_index_search_device(srs_index* index, const float* queries, int32_t q, int32_t dim, int32_t k,
                            const int32_t* exclude, int32_t* top_pos, float* top_scores, void* stream);
int srs_index_search_host(srs_index* index, const float* queries, int32_t q, int32_t dim, int32_t k,
                          const int32_t* exclude, int32_t* top_pos, float* top_scores);

/* One ranking call from host buffers: H2D of the candidate batch, forward kernel, ranking
 * kernel, D2H of the min(k, B) best positions and scores only.  Replaces
 * RecForYouProcess.ranker (:69-95) with model "nerualcf" followed by getRecList's subList:
 * the score vector never leaves the device.  Synchronous; SRS_ERR_RANGE as srs_predict_host. */
int srs_rank_host(srs_model* m, const srs_batch* batch, int32_t k, int32_t* top_idx,
                  float* top_scores);

/* ---- One ranking request "one user x n candidates" with the movie-side features resident in HBM.
 * The reference defines the serving feature store as Redis hashes `uf:<userId>` / `mf:<movieId>`
 * (FeatureEngForRecModel.scala:130-174,208-259; read at RecForYouProcess.java:46-52 and
 * DataManager.java:127-140).  srs_model_set_movie_features uploads the `mf:` side once: genres
 * [n_movies][3] as vocabulary indices (-1 = missing), numerics [n_movies][4] = movieAvgRating,
 * movieRatingCount, movieRatingStddev, releaseYear (already cast to float32).  A request then ships
 * one srs_user_row and n candidate ids - (9 + T + n) words instead of n full feature rows - and a
 * device kernel expands them into the batch the forward kernel reads (user columns broadcast, movie
 * columns gathered by candidate id).  srs_rank_user_host = that + forward + sort-and-cut
 * (RecForYouProcess.java:56-59), D2H of the best k positions / scores (and all n scores if
 * `probs` != NULL).  Candidate ids outside the table or the model's vocabulary give SRS_ERR_RANGE. */
typedef struct srs_user_row {
  int32_t user_id;
  int32_t user_genre[5];       /* userGenre1..5 vocabulary indices, -1 = missing                        */
  float user_numerics[3];      /* userAvgRating, userRatingCount, userRatingStddev                      */
  int32_t n_hist;              /* entries of `hist` (<= the model's history columns; the rest is id 0)  */
  const int32_t* hist;         /* userRatedMovie1.. in graph position order (most recent first)         */
} srs_user_row;
int srs_model_set_movie_features(srs_model* m, int32_t n_movies, const int32_t* genres,
                                 const float* numerics);
int srs_rank_user_host(srs_model* m, const srs_user_row* user, const int32_t* candidate_movie_ids,
                       int32_t n, int32_t k, int32_t* top_idx, float* top_scores, float* probs);

/* Debug aid for kernel tuning: enable/disable recording of per-phase SM-clock timestamps
 * in the tensor-core DIN kernels (CTA 0; slot meaning: profiles/trace_din_rt.py,
 * profiles/trace_din_tc.py) and, if out40 != NULL, synchronise and copy the 40 recorded values
 * out.  No effect on results. */
int srs_debug_din_trace(srs_model* m, int32_t enable, uint64_t* out40);

/* din_rtp_kernel only, with tracing enabled (srs_debug_din_trace): per-tile SM-clock timestamps of CTA 0,
 * out[kind * 64 + tile] (12 x 64 values), kinds 0 gather issued, 1 delivered, 2 weight operand built, 3 activation-unit
 * MMAs issued, 4 consumer sees the accumulators, 5 gate done, 6 pooling MMAs issued, 7 pooled rows read,
 * 8-11 inside the issuer (wait passed, MMAs issued, commits done, iteration start). */
int srs_debug_din_timeline(srs_model* m, uint64_t* out512);

/* Micro-benchmark behind the DIN kernel's MMA shape choice: SM cycles for a chain of n_mma
 * tcgen05.mma (M = 128, K = 16 bf16) with N in {32, 64, 128}, A from shared (0) or tensor (1)
 * memory, into one accumulator (two_acc bit 0 = 0) or alternating two (bit 0 = 1); bit 1 of
 * two_acc selects warp-uniform issue through elect.sync instead of a divergent single thread.
 * out2[0] = issue cycles, out2[1] = cycles until the commit barrier completes. */
int srs_debug_umma_bench(int32_t N, int32_t n_mma, int32_t a_in_tmem, int32_t two_acc,
                         int32_t device, uint64_t* out2);

/* Known-answer self test of the tcgen05 / TMEM plumbing the DIN kernel is built on:
 * D[128][N] = bf16(A[128][K]) * bf16(B[N][K])^T (inputs truncated to bf16, fp32 accumulate),
 * K = 64 * k_blocks (1..3), N = 16 or 32, A staged through shared memory (a_in_tmem = 0)
 * or written to tensor memory (a_in_tmem = 1).  Device pointers; synchronous. */
int srs_selftest_umma(const float* A, const float* B, float* D, int32_t N, int32_t k_blocks,
                      int32_t a_in_tmem, int32_t device);

#ifdef __cplusplus
}
#endif
#endif /* SRS_CTR_H_ */
