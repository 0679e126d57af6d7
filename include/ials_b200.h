/*
 * ials_b200.h -- C ABI of the B200-native iALS hot path (libials_b200.so).
 *
 * This is the drop-in boundary for irspack's native iALS core, i.e. for the
 * nanobind module `irspack.recommenders._ials_core`
 * (/root/reference/cpp_source/als/wrapper.cpp:17-182) and the C++ classes
 * behind it (cpp_source/als/IALSTrainer.hpp, IALSLearningConfig.hpp).  Every
 * entry point below names the reference interface it replaces.  Plain C:
 * opaque handle, plain pointers and sizes, no torch / C++ types.
 *
 * Conventions
 *   - All functions return an int status (IALS_OK == 0).  On failure
 *     ials_last_error() returns a thread-local message.  Status -> Python
 *     exception mapping mirrors the reference's C++ exceptions
 *     (cpp_source/argcheck.hpp:8-12, IALSTrainer.hpp:249-254, 317-323):
 *       IALS_ERR_INVALID_ARGUMENT -> ValueError   (std::invalid_argument)
 *       IALS_ERR_RUNTIME          -> RuntimeError (std::runtime_error)
 *       IALS_ERR_CUDA             -> RuntimeError
 *       IALS_ERR_NOT_IMPLEMENTED  -> NotImplementedError
 *   - "host" pointers are ordinary (pageable or pinned) host memory;
 *     "device" pointers live on the trainer's CUDA device.
 *   - Dense matrices crossing the boundary are row-major float32 with exactly K
 *     columns (Eigen RowMajor DenseMatrix, cpp_source/als/definitions.hpp:9-10).
 *     Inside the library rows are padded to `ld` floats: 128 for every K <= 128,
 *     round_up(K, 32) above.
 *   - CSR: int64 indptr[n_rows + 1], int32 indices[nnz] (ascending within a
 *     row), float data[nnz]  (Eigen::SparseMatrix<float, RowMajor>).
 *   - Calls on one handle are synchronous and not re-entrant, like the
 *     reference (it holds the GIL for the whole call).  Kernels run on the
 *     stream set with ials_trainer_set_stream (default: the legacy stream).
 *   - `side`: 0 = user, 1 = item.
 */
#ifndef IALS_B200_H
#define IALS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(IALS_BUILDING_LIBRARY) && defined(__GNUC__)
#define IALS_API __attribute__((visibility("default")))
#else
#define IALS_API
#endif

#define IALS_OK 0
#define IALS_ERR_INVALID_ARGUMENT 1
#define IALS_ERR_RUNTIME 2
#define IALS_ERR_CUDA 3
#define IALS_ERR_NOT_IMPLEMENTED 4

/* enum class LossType   { ORIGINAL, IALSPP }        IALSLearningConfig.hpp:11 */
#define IALS_LOSS_ORIGINAL 0
#define IALS_LOSS_IALSPP 1
/* enum class SolverType { Cholesky, CG, IALSPP }    IALSLearningConfig.hpp:12 */
#define IALS_SOLVER_CHOLESKY 0
#define IALS_SOLVER_CG 1
#define IALS_SOLVER_IALSPP 2

#define IALS_SIDE_USER 0
#define IALS_SIDE_ITEM 1
/* ials_trainer_similar */
#define IALS_SIMILARITY_DOT 0
#define IALS_SIMILARITY_COSINE 1

/* struct IALSModelConfig                            IALSLearningConfig.hpp:15-31 */
typedef struct ials_model_config {
  int64_t K;
  float alpha0;
  float reg;
  float nu;
  float init_stdev;
  int32_t random_seed;
  int32_t loss_type;
} ials_model_config;

/* struct SolverConfig                               IALSLearningConfig.hpp:97-112 */
typedef struct ials_solver_config {
  int64_t n_threads;    /* validated (> 0) like the reference, otherwise unused on GPU */
  int32_t solver_type;
  int32_t reserved;
  int64_t max_cg_steps; /* 0 means K, IALSTrainer.hpp:232-234 */
  int64_t ialspp_subspace_dimension;
  int64_t ialspp_iteration;
} ials_solver_config;

typedef struct ials_trainer ials_trainer;

/* Thread-local message of the last failing call on this thread. */
IALS_API const char *ials_last_error(void);
/* "major.minor.patch" of this library. */
IALS_API const char *ials_version(void);
/* Number of visible CUDA devices (0 if none / no driver). */
IALS_API int ials_device_count(void);

/* IALSTrainer::IALSTrainer(config, X)                IALSTrainer.hpp:710-720
 * Copies X (host CSR, n_users x n_items) to `device`, builds X^T there, and
 * initialises both factor matrices with std::mt19937(random_seed) +
 * std::normal_distribution<float>(0, init_stdev / sqrt(K))  (:64-76). */
IALS_API int ials_trainer_create(const ials_model_config *config, int64_t n_users, int64_t n_items,
                        const int64_t *indptr, const int32_t *indices, const float *data,
                        int device, ials_trainer **out);

/* Same, but the CSR arrays already live in device memory (they are copied;
 * the caller keeps ownership).  Used for matrices generated on the GPU.
 * `init_on_device` != 0 replaces the serial host RNG by a counter-based device
 * generator with the same distribution (for very large factor matrices). */
IALS_API int ials_trainer_create_from_device_csr(const ials_model_config *config, int64_t n_users,
                                        int64_t n_items, const int64_t *d_indptr,
                                        const int32_t *d_indices, const float *d_data,
                                        int device, int init_on_device, ials_trainer **out);

/* IALSTrainer::IALSTrainer(config, user, item)  "used when deserialize"
 *                                                    IALSTrainer.hpp:745-756
 * No interaction matrix: the trainer can score and fold in, but step() fails
 * with IALS_ERR_RUNTIME. */
IALS_API int ials_trainer_create_from_factors(const ials_model_config *config, int64_t n_users,
                                     int64_t n_items, const float *user, const float *item,
                                     int device, ials_trainer **out);

IALS_API void ials_trainer_destroy(ials_trainer *t);

/* Stream all subsequent work of this trainer is enqueued on (a cudaStream_t). */
IALS_API int ials_trainer_set_stream(ials_trainer *t, void *cuda_stream);

/* IALSTrainer::step(solver_config)                   IALSTrainer.hpp:758-789
 * One epoch: Gram(item) -> solve users -> Gram(user) -> solve items.
 * Synchronises and reports solver failures (singular CG system, failed
 * Cholesky) as IALS_ERR_RUNTIME with the reference's messages. */
IALS_API int ials_trainer_step(ials_trainer *t, const ials_solver_config *solver);

/* The same epoch, enqueued without the trailing synchronisation / error check
 * (for back-to-back epochs and device-side timing).  ials_trainer_sync()
 * waits and reports any solver failure recorded since the last sync. */
IALS_API int ials_trainer_step_async(ials_trainer *t, const ials_solver_config *solver);

/* One epoch on HOST-resident factors (what `trainer.user = u; trainer.item = v;
 * trainer.step(cfg); u = trainer.user; v = trainer.item` does through
 * wrapper.cpp:137,158-159, as one call): uploads item_in and user_in
 * (C-contiguous float32 [n x K]; pinned memory makes the copies asynchronous),
 * runs the epoch, and writes the new factors to user_out / item_out.  The user
 * matrix travels back on a second stream while the item half-epoch runs.
 * Synchronises and reports solver failures like ials_trainer_step. */
IALS_API int ials_trainer_step_io(ials_trainer *t, const ials_solver_config *solver,
                                  const float *user_in, const float *item_in, float *user_out,
                                  float *item_out);
IALS_API int ials_trainer_sync(ials_trainer *t);

/* Half an epoch: Solver::prepare_p + Solver::step for one side
 * (IALSTrainer.hpp:78-115 + 664-679).  side 0 solves users against items. */
IALS_API int ials_trainer_half_step(ials_trainer *t, int side, const ials_solver_config *solver);

/* Solver::prepare_p result for `side`: out[K*K] = alpha0 * Y^T Y with Y the
 * OTHER side's factors (user_solver.P is built from item).  :78-115 */
IALS_API int ials_trainer_gram(ials_trainer *t, int side, float *out_host);

/* IALSTrainer::user_scores(begin, end, solver_config) IALSTrainer.hpp:942-984
 * out_host[(end-begin) * n_items], row-major. */
IALS_API int ials_trainer_user_scores(ials_trainer *t, int64_t begin, int64_t end,
                             const ials_solver_config *solver, float *out_host);

/* def_rw("user") / def_rw("item")                    wrapper.cpp:158-159 */
IALS_API int ials_trainer_get_factors(ials_trainer *t, int side, float *out_host);
IALS_API int ials_trainer_set_factors(ials_trainer *t, int side, const float *in_host);
/* The same for the rows [row_begin, row_begin + n_rows) only (host buffer n_rows x K).  On a
 * row-sharded trainer with push_to_peers != 0 the uploaded rows are then copied device to
 * device into every peer's replica (CUDA IPC over NVLink): each rank brings ITS OWN rows down
 * from the host, the peers receive them over the fabric.  Asynchronous on the trainer's stream
 * (the host buffer must stay valid until ials_trainer_sync); the peers' copies are ordered
 * before their next solve by the Gram all-reduce, like the solve kernels' peer stores. */
IALS_API int ials_trainer_set_factor_rows(ials_trainer *t, int side, int64_t row_begin, int64_t n_rows,
                                          const float *in_host, int push_to_peers);
/* Upload of the user rows this trainer solves (the whole matrix, or a rank's shard) that OVERLAPS
 * the next user half-epoch: the rows arrive in 2 MB chunks on a copy stream, the copy engine
 * raises a flag behind each, and the CG kernels of the 128-column layout read a row's flag before
 * its warm start (any other solve waits for the whole upload first).  The rows are NOT pushed to
 * peer replicas: they are warm starts, the solve kernels store the new values everywhere.  The
 * host buffer must stay valid until the next synchronising call. */
IALS_API int ials_trainer_set_user_rows_flagged(ials_trainer *t, int64_t row_begin, int64_t n_rows,
                                                const float *in_host);
IALS_API int ials_trainer_get_factor_rows(ials_trainer *t, int side, int64_t row_begin, int64_t n_rows,
                                          float *out_host);
/* Zero-copy access for on-device consumers (torch views, NCCL): base pointer,
 * row count, K and row stride (in floats) of the padded device matrix. */
IALS_API int ials_trainer_factors_device(ials_trainer *t, int side, float **d_ptr, int64_t *n_rows,
                                int64_t *K, int64_t *ld);

/* IALSTrainer::transform_user / transform_item       IALSTrainer.hpp:791-802
 * side 0: X is (n_rows x n_items), returns n_rows x K user vectors.
 * side 1: X is (n_users x n_cols) exactly as the reference takes it (it is
 *         transposed inside, :800), returns n_cols x K item vectors.
 * Shape mismatch -> IALS_ERR_INVALID_ARGUMENT (Solver::X_to_vector :126-131). */
IALS_API int ials_trainer_transform(ials_trainer *t, int side, int64_t n_rows, int64_t n_cols,
                           const int64_t *indptr, const int32_t *indices, const float *data,
                           const ials_solver_config *solver, float *out_host);

/* ---- Feature-aware iALS ------------------------------------------------------------------
 * IALSTrainer(model_config, interaction, user_feature, item_feature)   wrapper.cpp:133-136,
 * IALSTrainer.hpp:722-743.  A feature matrix is dense row-major (indptr == NULL) or CSR
 * [n_rows x n_cols]; n_cols may be 0 (that side then trains as plain iALS).
 *
 * ials_trainer_set_features: call once per side right after ials_trainer_create, with
 * config.lambda_{user,item}_feature and config.feature_warmup_epochs (the same value for both sides).
 * Errors of initialize_feature_aware (:1001-1014): "Feature matrix row count mismatch.",
 * "Feature weight regularization must be positive."  From then on ials_trainer_step[_async|_io] is
 * IALSTrainer::step of the feature-aware model (:758-789): after the warm-up epochs a side with
 * features is solved towards its prior  features x weight  (Solver::step_with_prior :634-662, CG
 * or Cholesky; IALSPP -> "Feature-aware iALS does not support IALSPP.") and its weight is refit
 * by the weighted ridge regression of :1066-1209 ("Feature ridge Cholesky decomposition
 * failed." / "Feature ridge solve failed." surface at the next synchronising call). */
IALS_API int ials_trainer_set_features(ials_trainer *t, int side, int64_t n_rows, int64_t n_cols,
                                       const float *dense, const int64_t *indptr, const int32_t *indices,
                                       const float *data, float lambda_feature, int64_t feature_warmup_epochs);
/* user_feature_weight / item_feature_weight (def_rw, wrapper.cpp:160-161): [rows x K] row-major;
 * rows = 0 for a trainer without features. */
IALS_API int ials_trainer_feature_weight_rows(ials_trainer *t, int side, int64_t *n_rows);
IALS_API int ials_trainer_get_feature_weight(ials_trainer *t, int side, float *out_host);
IALS_API int ials_trainer_set_feature_weight(ials_trainer *t, int side, int64_t n_rows, const float *in_host);
/* transform_user_feature / transform_item_feature (:820-830): out [n_rows x K] = features x weight.
 * "... feature weights are not initialized." / "Shape mismatch: ..." as :1016-1042. */
IALS_API int ials_trainer_transform_feature(ials_trainer *t, int side, int64_t n_rows, int64_t n_cols,
                                            const float *dense, const int64_t *indptr, const int32_t *indices,
                                            const float *data, float *out_host);
/* transform_user_with_feature / transform_item_with_feature (:803-818): the fold-in of
 * ials_trainer_transform whose rows start from, and are regularised towards, features x weight
 * (X_to_vector_with_prior :142-167); the feature matrix has one row per NEW row. */
IALS_API int ials_trainer_transform_with_feature(ials_trainer *t, int side, int64_t n_rows, int64_t n_cols,
                                                 const int64_t *indptr, const int32_t *indices, const float *data,
                                                 int64_t f_rows, int64_t f_cols, const float *f_dense,
                                                 const int64_t *f_indptr, const int32_t *f_indices,
                                                 const float *f_data, const ials_solver_config *solver,
                                                 float *out_host);

/* IALSTrainer::compute_loss(solver_config)           IALSTrainer.hpp:836-940 */
IALS_API int ials_trainer_compute_loss(ials_trainer *t, const ials_solver_config *solver, float *out);

/* Fused replacement of the Evaluator's scoring chunk:
 *   get_score_block (ials.py:483-484 -> IALSTrainer.hpp:942-984)
 *   + scores[mask.nonzero()] = -inf (evaluation/evaluator.py:426-432)
 *   + top-`k` by (-score, index)     (cpp_source/evaluator.cpp:324-355)
 * for users [begin, end).  mask_mode: 0 = rows of the training matrix X,
 * 1 = no mask, 2 = host CSR (mask_indptr has end-begin+1 entries, relative to
 * `begin`; stored zeros must already be removed, as scipy's .nonzero() does).
 * out_idx[(end-begin)*k] (-1 padded), out_score (same shape, may be NULL),
 * out_count[end-begin] = number of valid entries per user. */
IALS_API int ials_trainer_recommend(ials_trainer *t, int64_t begin, int64_t end, int64_t k,
                           int mask_mode, const int64_t *mask_indptr,
                           const int32_t *mask_indices, int32_t *out_idx, float *out_score,
                           int32_t *out_count);
/* The same with allow-lists fused into the kernel's epilogue (recommendable items of the Evaluator,
 * evaluator.py:115-136; allowed_item_indices of retrieve_recommend_from_score, util.hpp:426-504):
 * allow_n_lists = 1 (one list for every row) or end - begin (one per row), CSR with int32 item ids
 * strictly ascending inside a list.  Only items on a row's list can be returned (seen / masked items
 * are still dropped).  No score block ever leaves the device.  Needs the fused kernel (any row
 * stride, k <= 128, mask rows strictly ascending), otherwise IALS_ERR_NOT_IMPLEMENTED. */
IALS_API int ials_trainer_recommend_allowed(ials_trainer *t, int64_t begin, int64_t end, int64_t k, int mask_mode,
                                            const int64_t *mask_indptr, const int32_t *mask_indices,
                                            int64_t allow_n_lists, const int64_t *allow_indptr,
                                            const int32_t *allow_indices, int32_t *out_idx, float *out_score,
                                            int32_t *out_count);
/* The serving form (IDMapper.recommend_for_known_user_batch, utils/id_mapping.py:418-453: get_score_remove_seen
 * of arbitrary user indices -> forbidden items -> retrieve_recommend_from_score, util.hpp:426-504) without a
 * host score block: the users are picked by index (any order, repeats allowed), their factor rows are
 * gathered on the device and go through the same fused kernel.  mask_mode 0 hides each user's own
 * training row; mask_mode 2 takes one CSR row per listed user (e.g. training row + forbidden items);
 * allow-lists as in ials_trainer_recommend_allowed (allow_n_lists = 0: none).  out_score holds the
 * scores of the returned items. */
IALS_API int ials_trainer_recommend_users(ials_trainer *t, const int64_t *user_indices, int64_t n_users, int64_t k,
                                          int mask_mode, const int64_t *mask_indptr, const int32_t *mask_indices,
                                          int64_t allow_n_lists, const int64_t *allow_indptr,
                                          const int32_t *allow_indices, int32_t *out_idx, float *out_score,
                                          int32_t *out_count);
/* The same for users that are not rows of the model: user_embeddings[n_rows * K] (host, row-major; what
 * ials_trainer_transform returns for new users' profiles -- get_score_cold_user / get_score_from_user_embedding,
 * recommenders/ials.py:486-490, 529-533) are scored against the trainer's item factors where they lie on
 * the device.  mask_mode 1 (none) or 2 (one CSR row per embedding, e.g. the profile itself). */
IALS_API int ials_trainer_recommend_embeddings(ials_trainer *t, const float *user_embeddings, int64_t n_rows,
                                               int64_t k, int mask_mode, const int64_t *mask_indptr,
                                               const int32_t *mask_indices, int64_t allow_n_lists,
                                               const int64_t *allow_indptr, const int32_t *allow_indices,
                                               int32_t *out_idx, float *out_score, int32_t *out_count);
/* Nearest neighbours within one side (new: the reference has no such query): for each query row of
 * `side` (0: similar users, 1: similar items), the best `k` rows of the same side, ordered by
 * (-score, index) as the lists above.  Queries: query_idx[0 .. end) (host, any order, repeats allowed;
 * begin must be 0) or, with query_idx null, the rows [begin, end) of the side.  metric
 * IALS_SIMILARITY_COSINE: q.y / (|q| |y|), 0 when either row is zero (the side is copied at unit norm on
 * every call); IALS_SIMILARITY_DOT: q.y.  exclude_self hides the query row itself; forbid_indptr /
 * forbid_indices (optional host CSR, one row per query, any order) hide more rows; allow-lists as in
 * ials_trainer_recommend_allowed, over the side's rows.  1 <= k <= min(1024, rows of the side); k <= 128
 * runs the fused tensor-core kernel, larger k dense scores + SIMT top-k (allow-lists: k <= 128 only,
 * IALS_ERR_NOT_IMPLEMENTED otherwise).  Lists shorter than k are padded with -1 (out_count: their
 * lengths); out_score (optional) holds the scores.  No trainer state changes. */
IALS_API int ials_trainer_similar(ials_trainer *t, int side, const int64_t *query_idx, int64_t begin, int64_t end,
                                  int64_t k, int metric, int exclude_self, const int64_t *forbid_indptr,
                                  const int32_t *forbid_indices, int64_t allow_n_lists, const int64_t *allow_indptr,
                                  const int32_t *allow_indices, int32_t *out_idx, float *out_score,
                                  int32_t *out_count);
/* Candidate ranking (new: the reference ranks allowed items by computing every item's score first):
 * for each query row, the best `k` items of its own candidate list by the score q . item, ordered by
 * (-score, index) as the lists above.  The cost follows the number of (row, candidate) pairs, not the
 * catalogue: the candidates' item rows are gathered and dotted in FP32, and each list is selected on
 * its own.  Queries: user_idx[0 .. end) (host, any order, repeats allowed; begin must be 0), or
 * user_emb[end * K] (host embeddings, e.g. fold-in results; begin must be 0), or, with both null, the
 * users [begin, end); both non-null is an error.  mask_mode as in ials_trainer_recommend_users (0: each
 * user's training row, not with embeddings and, on a row-sharded trainer, only for the rank's own users;
 * 1: none; 2: one host CSR row per query).  Candidates: a CSR of int32 item ids, one list shared by
 * every row (cand_n_lists = 1) or one per row (cand_n_lists = end - begin), each list strictly ascending
 * in [0, n_items).  1 <= k <= min(1024, n_items).  Masked candidates are dropped; lists shorter than k
 * are padded with -1 (scores -inf), out_count holds their lengths, out_score may be NULL.  Rows run in
 * slabs whose lists are copied to the host one after the other.  Every invalid argument is
 * IALS_ERR_INVALID_ARGUMENT.  No trainer state changes. */
IALS_API int ials_trainer_rank_candidates(ials_trainer *t, const int64_t *user_idx, const float *user_emb,
                                          int64_t begin, int64_t end, int64_t k, int mask_mode,
                                          const int64_t *mask_indptr, const int32_t *mask_indices,
                                          int64_t cand_n_lists, const int64_t *cand_indptr,
                                          const int32_t *cand_indices, int32_t *out_idx, float *out_score,
                                          int32_t *out_count);
/* The scores alone ("predict" of the factor model, or iALS scores as features of another ranker):
 * out_scores[j] = q_r . item[cand_indices[j]] in FP32 for every entry j of row r of the CSR
 * cand_indptr[end - begin + 1] / cand_indices (any order, repeats allowed, ids in [0, n_items)), in
 * input order.  Queries as in ials_trainer_rank_candidates.  No mask, no selection. */
IALS_API int ials_trainer_candidate_scores(ials_trainer *t, const int64_t *user_idx, const float *user_emb,
                                           int64_t begin, int64_t end, const int64_t *cand_indptr,
                                           const int32_t *cand_indices, float *out_scores);
/* Explanations (new; Hu, Koren and Volinsky, ICDM 2008, section 5, and `implicit`'s ALS.explain): why a
 * row of `side` (0: users) scores a target row t of the other side.  With Y the other side's factors,
 * P = alpha0 Y^T Y (recomputed from Y on every call, into the side's P), the row's history (j, c_j),
 * reg_u = reg (alpha0 n_other + nnz_u)^nu, bias = alpha0 (ORIGINAL) or 0 (IALSPP) and prior_u the stored
 * feature prior F W (rows by index past the warm-up epochs only):
 *   A_u = P + sum_j c_j y_j y_j^T + reg_u I,  x_u = A_u^-1 (sum_j (bias + c_j) y_j + reg_u prior_u),
 *   w_t = A_u^-1 y_t,  score = y_t . x_u = sum_j (bias + c_j) w_t . y_j + reg_u w_t . prior_u.
 * Per (query row, target) pair: out_score = y_t . x_u, out_prior (optional) = reg_u w_t . prior_u, and
 * the best n_top history entries by contribution (bias + c_j) w_t . y_j, ordered by (-contribution,
 * column id), as column ids (out_idx [pairs x n_top], padded with -1) and contributions (out_contrib,
 * optional, padded with -inf), out_count = min(n_top, history length).  Every stored entry counts (stored
 * zeros, repeated columns).  A row with an empty history and no prior gives 0, 0 and count 0.
 * Queries: query_idx[0 .. end) (host, any order, repeats allowed, begin = 0), or a host CSR of `end` cold
 * rows hist_indptr / hist_indices / hist_data over the other side's ids (begin = 0, no prior), or, with
 * all of them null, the rows [begin, end).  On a row-sharded trainer rows by index must be the rank's own.
 * Targets: a host CSR of one list per query row (any order, repeats allowed, ids in [0, n_other)); the
 * pairs come out in its order.  1 <= n_top <= 1024.  A failed factorisation raises "Cholesky decomposition
 * failed." (IALS_ERR_RUNTIME); K > 256 is IALS_ERR_NOT_IMPLEMENTED; every invalid argument is
 * IALS_ERR_INVALID_ARGUMENT.  The factors do not change. */
IALS_API int ials_trainer_explain(ials_trainer *t, int side, const int64_t *query_idx, int64_t begin, int64_t end,
                                  const int64_t *hist_indptr, const int32_t *hist_indices, const float *hist_data,
                                  const int64_t *target_indptr, const int32_t *target_indices, int64_t n_top,
                                  float *out_score, float *out_prior, int32_t *out_idx, float *out_contrib,
                                  int32_t *out_count);

/* Mask + top-`k` for a block of precomputed float32 scores (any recommender;
 * replaces EvaluatorCore::get_metrics_local's selection, evaluator.cpp:324-355,
 * plus the mask scatter of evaluator.py:426-432).  scores_host[rows * n_items];
 * mask CSR is optional (both NULL = no mask), relative to the block. */
IALS_API int ials_topk_scores(const float *scores_host, int64_t rows, int64_t n_items, int64_t k,
                     const int64_t *mask_indptr, const int32_t *mask_indices, int device,
                     void *cuda_stream, int32_t *out_idx, float *out_score, int32_t *out_count);

/* Metrics::update over a block of users            cpp_source/evaluator.cpp:127-166, 308-361
 * (get_metrics_local's per-user bookkeeping, given the lists the selection produced):
 * rec[rows * k] item indices (-1 padded), count[rows] valid entries, the block's ground truth as a
 * CSR with sorted rows, discount[k] = 1 / log2(2 + j) (prepare_dcg_discount, :42-48).  ADDS to
 * acc[5] = {hit, recall, ndcg, map, precision} sums over valid users, *valid_user and
 * item_cnt[n_items] (the caller's Metrics accumulator).  One warp per user on the device. */
IALS_API int ials_metrics_accumulate(const int32_t *rec, const int32_t *count, int64_t rows, int64_t k,
                                     const int64_t *gt_indptr, const int32_t *gt_indices, int64_t n_items,
                                     int recall_with_cutoff, const double *discount, int device,
                                     void *cuda_stream, double *acc, int64_t *valid_user, int64_t *item_cnt);

/* ---- evaluation passes that keep the lists on the device ----
 * An evaluation set holds, on the trainer's device, everything an Evaluator pass needs besides the
 * model: the ground-truth rows of users [row_begin, row_begin + n_rows) (CSR from 0, rows sorted
 * ascending; host arrays, or device arrays with gt_on_device != 0, which are copied), the mask (both
 * mask pointers NULL: the trainer's training rows, as the Evaluator's "train"; else a host CSR of
 * n_rows rows without stored zeros), the allow-lists of ials_trainer_recommend_allowed (allow_n_lists
 * 0, 1 or n_rows; rows relative to row_begin; they need the fused kernel: every cutoff <= 128, else
 * IALS_ERR_NOT_IMPLEMENTED), the cutoffs (each in [1, n_items], <= 1024), recall_with_cutoff, and
 * per cutoff the accumulators of Metrics::update (cpp_source/evaluator.cpp:127-166): five float64 sums,
 * valid_user / total_user and the item-count histogram.  Uploaded once. */
typedef struct ials_eval_set ials_eval_set;
IALS_API int ials_eval_set_create(ials_trainer *t, int64_t row_begin, int64_t n_rows, const int64_t *gt_indptr,
                                  const int32_t *gt_indices, int gt_on_device, const int64_t *mask_indptr,
                                  const int32_t *mask_indices, int64_t allow_n_lists, const int64_t *allow_indptr,
                                  const int32_t *allow_indices, const int64_t *cutoffs, int64_t n_cutoffs,
                                  int recall_with_cutoff, ials_eval_set **out);
IALS_API void ials_eval_set_destroy(ials_eval_set *e);
/* Zeroes the accumulators on `cuda_stream`. */
IALS_API int ials_eval_set_reset(ials_eval_set *e, void *cuda_stream);
/* Device pointers of the accumulators, for an all-reduce in place: sums[n_cutoffs][5] (float64 hit,
 * recall, ndcg, map, precision), counts[2][n_cutoffs] (int64 valid_user, then total_user) and
 * hist[n_cutoffs][n_items] (int64). */
IALS_API int ials_eval_set_buffers(ials_eval_set *e, double **sums, int64_t **counts, int64_t **hist,
                                   int64_t *n_cutoffs, int64_t *n_items);
/* out[n_cutoffs][3] = {appeared_item, entropy, gini_index} of each histogram, as Metrics::as_dict
 * (:87-123) computes them, on the device without sorting; synchronous. */
IALS_API int ials_eval_set_diversity(ials_eval_set *e, void *cuda_stream, double *out);
/* One evaluation pass over users [user_begin, user_end) (inside the set's rows and, with the training
 * mask, inside the rank's shard): the lists of ials_trainer_recommend[_allowed] with k = max(cutoffs),
 * in chunks, each followed by the metrics kernel, on the trainer's stream; ADDS to the accumulators.
 * The sums are deterministic: the same pass gives the same bits.  Returns when the pass is done. */
IALS_API int ials_trainer_evaluate(ials_trainer *t, ials_eval_set *e, int64_t user_begin, int64_t user_end);
/* A cold evaluation set (EvaluatorWithColdUser, evaluation/evaluator.py:470-657): n_rows users that are
 * not rows of the model.  Their input rows (CSR [n_rows x n_cols], n_cols == n_items, else "Shape mismatch:
 * ..." as Solver::X_to_vector :126-131) are what the fold-in solves, as given: stored zeros count in nnz and
 * add bias * y.  The mask (both mask pointers NULL) is the input's non-zeros, as scipy's .nonzero() gives
 * them (evaluator.py:432); a host CSR of n_rows rows without stored zeros replaces it (masked_interactions,
 * evaluator.py:574-577).  Ground truth, allow-lists (rows relative to the set), cutoffs and accumulators as
 * in ials_eval_set_create.  The input and ground-truth arrays are host arrays, or device arrays with
 * on_device != 0; the input is validated and planned once, in chunks of the pass. */
IALS_API int ials_eval_set_create_cold(ials_trainer *t, int64_t n_rows, int64_t n_cols, const int64_t *in_indptr,
                                       const int32_t *in_indices, const float *in_data, const int64_t *gt_indptr,
                                       const int32_t *gt_indices, int on_device, const int64_t *mask_indptr,
                                       const int32_t *mask_indices, int64_t allow_n_lists, const int64_t *allow_indptr,
                                       const int32_t *allow_indices, const int64_t *cutoffs, int64_t n_cutoffs,
                                       int recall_with_cutoff, ials_eval_set **out);
/* One pass over the cold set's rows [row_begin, row_end), on the trainer's stream with one synchronisation
 * at the end: P = alpha0 item^T item of the full item factors once, then per chunk the fold-in of
 * ials_trainer_transform (side 0, from zero, every solver route of `solver`) into a device slab, the lists
 * of ials_trainer_evaluate on that slab and the metrics of every cutoff; ADDS to the accumulators.  No
 * training state changes.  Solver failures raise with the reference's messages (IALSTrainer.hpp:252-253,
 * 318, 322).  A row-sharded trainer runs it on its own share of the cold users; its item factors are a
 * full replica, so the pass needs no collective. */
IALS_API int ials_trainer_evaluate_cold(ials_trainer *t, ials_eval_set *e, const ials_solver_config *solver,
                                        int64_t row_begin, int64_t row_end);

/* retrieve_recommend_from_score<float>                 cpp_source/util.hpp:426-504
 * (bound as irspack.utils._util_cpp.retrieve_recommend_from_score_f32,
 * cpp_source/util.cpp; caller: utils/id_mapping.py:29-46, 297-324).
 * For every row of scores_host[rows * n_items]: the candidates are all items,
 * or the row's allow-list (out-of-range and negative entries are ignored,
 * util.hpp:466-469); the best `cutoff` by descending score are returned, items
 * scored -inf never (:489-491).  Ties are returned in ascending index order
 * (the reference's comparator leaves them unspecified); a duplicate in an
 * allow-list is one candidate.
 * n_allowed_lists: 0 = no restriction, 1 = allowed_indptr[0..1] shared by all
 * rows, rows = one list per row; anything else -> IALS_ERR_INVALID_ARGUMENT
 * with the reference's message (:436-439).  cutoff is clamped to n_items;
 * cutoff > 1024 -> IALS_ERR_NOT_IMPLEMENTED.
 * out_idx[rows * min(cutoff, n_items)] (-1 padded), out_score likewise (may be
 * NULL), out_count[rows]. */
IALS_API int ials_retrieve_recommend(const float *scores_host, int64_t rows, int64_t n_items,
                            int64_t cutoff, int64_t n_allowed_lists,
                            const int64_t *allowed_indptr, const int64_t *allowed_indices,
                            int device, void *cuda_stream, int32_t *out_idx, float *out_score,
                            int32_t *out_count);

/* Tensor-core operator behind Solver::prepare_p (IALSTrainer.hpp:78-115) and the
 * rank updates of Solver::step_cholesky (:37-58, 301-308):
 *   G[K*K] = sum_{t<m} w[t] * y_{idx[t]} y_{idx[t]}^T,   b[K] = sum_t (bias + w[t]) * y_{idx[t]}
 * Y is n x K row-major (K <= 128).  idx == NULL: all n rows in order (m ignored);
 * w == NULL: unit weights; weights must be >= 0.  The sum is split into n_jobs
 * contiguous jobs (one persistent CTA each) whose partials are added in job order.
 * Computed with tcgen05.mma kind::tf32 on an error-compensated hi/lo split
 * (fp32-level accuracy: see irspack_b200/csrc/wgram.cu).  b may be NULL. */
IALS_API int ials_weighted_gram(const float *Y_host, int64_t n, int64_t K, const int32_t *idx_host,
                       const float *w_host, int64_t m, int64_t n_jobs, float bias, int device,
                       float *G_host, float *b_host);

/* The same operator for 256-column factors (128 < K <= 256; the rank updates of the K = 256
 * Cholesky solver, BatchedRankUpdater IALSTrainer.hpp:37-58): the one-pass 256 x 256 tensor-core
 * kernel (W = 1/2 hi (hi + 2 lo)^T per job, G = W + W^T), assembled into G_host[K*K] and b_host[K]. */
IALS_API int ials_weighted_gram256(const float *Y_host, int64_t n, int64_t K, const int32_t *idx_host,
                          const float *w_host, int64_t m, int64_t n_jobs, float bias, int device,
                          float *G_host, float *b_host);

/* Both operators job by job (K <= 256): job j sums the entries [job_begin[j], job_end[j]) of
 * (idx, w) -- of the rows of Y when idx is NULL (m ignored) -- in one launch of the K <= 128
 * kernel (row stride 128) or of the 256-column one (128 < K <= 256), and returns its own block
 *   G_jobs[j][K*K] = W_j + W_j^T,   b_jobs[j][K] = sum_{t in job j} (bias + w[t]) * y_{idx[t]}
 * Any bounds with 0 <= begin <= end <= m are accepted: empty, overlapping or out-of-order jobs.
 * n_jobs <= 4096 (K <= 128) or 1024 (K > 128); m <= 2^31 - 64; b_jobs may be NULL. */
IALS_API int ials_weighted_gram_jobs(const float *Y_host, int64_t n, int64_t K, const int32_t *idx_host,
                            const float *w_host, int64_t m, const int64_t *job_begin,
                            const int64_t *job_end, int64_t n_jobs, float bias, int device,
                            float *G_jobs, float *b_jobs);

/* Device-side phase timing.  When enabled, every epoch enqueued by
 * ials_trainer_step[_async] records CUDA events (on the trainer's stream)
 * around its phases.  ials_trainer_get_timings synchronises, adds up the elapsed
 * milliseconds since the last call into
 *   ms[0] Gram(item)   users: ms[1] tensor-core Gram of heavy rows, ms[2] their dense CG,
 *                             ms[3] all other rows (the whole solve for Cholesky)
 *   ms[4] Gram(user)   items: ms[5], ms[6], ms[7] likewise
 * and returns the number of epochs covered in *n_epochs. */
IALS_API int ials_trainer_set_profiling(ials_trainer *t, int enabled);
IALS_API int ials_trainer_get_timings(ials_trainer *t, double ms[8], int64_t *n_epochs);
/* Row schedule of `side` (0: users = rows of X, 1: items = rows of X^T):
 * out = { rows, nnz, heavy rows, nnz in heavy rows, tensor-core jobs, max degree,
 *         hot columns cached in shared memory by the light-row kernel, per-mille of the
 *         light rows' entries that gather one of them }.
 * Heavy rows (degree > IALS_HEAVY_THRESHOLD, default 2048, K padded to 128 only) form
 * their normal equations explicitly on the tensor cores. */
IALS_API int ials_trainer_plan_stats(ials_trainer *t, int side, int64_t out[8]);
/* Number of CUDA kernels this library has launched in this process so far. */
IALS_API int64_t ials_kernel_launch_count(void);

/* ---- row-sharded multi-GPU (one process per GPU; new design, SURVEY.md 8e) ---- */

/* One rank of a row-sharded trainer.  The reference has no multi-process path;
 * this partitions the row-parallel loops of Solver::step (IALSTrainer.hpp:180-270,
 * 278-330: every worker writes only its own target rows) across GPUs.  The rank
 * owns users [user_begin, user_end) and items [item_begin, item_end): it receives
 * ONLY those rows of X (u_* arrays: user_end-user_begin+1 indptr entries starting
 * at 0, column = global item id) and of X^T (i_* arrays, column = global user id),
 * keeps full replicas of both factor matrices, and solves only its own rows.
 * csr_on_device != 0: the six CSR arrays are device pointers (copied).
 * An epoch is driven by the caller (irspack_b200/dist.py):
 *   for side in (user, item):
 *     ials_trainer_gram_partial(1 - side) -> all-reduce(sum) the K*K buffer
 *     ials_trainer_solve_shard(side)       (writes local + peer replicas)
 * (the feature-aware epoch adds a refit per side, see below).
 * ials_trainer_step / half_step / compute_loss refuse a sharded trainer. */
IALS_API int ials_trainer_create_sharded(const ials_model_config *config, int64_t n_users,
                                int64_t n_items, int64_t user_begin, int64_t user_end,
                                const int64_t *u_indptr, const int32_t *u_indices,
                                const float *u_data, int64_t item_begin, int64_t item_end,
                                const int64_t *i_indptr, const int32_t *i_indices,
                                const float *i_data, int csr_on_device, int init_on_device,
                                int device, ials_trainer **out);
/* Rows of `side` this trainer solves ([0, n) for an unsharded trainer). */
IALS_API int ials_trainer_shard_range(ials_trainer *t, int side, int64_t *begin, int64_t *end);
/* Partial Gram alpha0 * Y_shard^T Y_shard of this rank's own rows of `factor_side`
 * (Solver::prepare_p restricted to the shard, IALSTrainer.hpp:78-115)
 * written to a device K*K (ld-padded: ld*ld floats) buffer owned by the trainer;
 * the caller all-reduces it in place and calls ials_trainer_solve_shard. */
IALS_API int ials_trainer_gram_partial(ials_trainer *t, int factor_side, float **d_out, int64_t *count);
/* Solve this rank's rows of `side` using the (already all-reduced) Gram buffer
 * of the other side; writes the rows into the local replica and, if peer
 * replicas were registered, into every peer's replica as well.  A side that uses
 * its features (set with ials_trainer_set_shard_features, past the warm-up) is
 * solved towards the prior features x weight of the shard's rows, as
 * ials_trainer_step does (IALSTrainer.hpp:762-787), and its weight refit becomes due.
 * The item side (side 1) ends the epoch: it advances the epoch counter that the
 * warm-up is measured in (:788). */
IALS_API int ials_trainer_solve_shard(ials_trainer *t, int side, const ials_solver_config *solver);

/* ---- feature-aware iALS on a row-sharded trainer ----
 * The feature-aware epoch of IALSTrainer::step (:758-789) across ranks.  Per side:
 *   ials_trainer_gram_partial(1 - side) -> all-reduce
 *   ials_trainer_solve_shard(side)             (prior F_own W when the side uses features)
 *   ials_trainer_feature_partials(side) -> all-reduce each buffer with a non-zero count
 *   ials_trainer_feature_refit(side)           (every rank solves the same summed system)
 * The weights stay identical on every rank; ials_trainer_get_feature_weight /
 * _set_feature_weight read and write this rank's copy. */
/* IALSTrainer(config, X, user_feature, item_feature) for this rank's rows of `side`
 * (initialize_feature_aware :1001-1014): n_rows = the shard's rows, dense or CSR, the arguments
 * and errors of ials_trainer_set_features.  *has_empty_row (may be NULL) reports whether one of
 * the shard's rows of X (side 0) / X^T (side 1) is empty: the guard of step_with_prior
 * (:639-652) needs the OR over all ranks, see ials_trainer_check_shard_step. */
IALS_API int ials_trainer_set_shard_features(ials_trainer *t, int side, int64_t n_rows, int64_t n_cols,
                                             const float *dense, const int64_t *indptr, const int32_t *indices,
                                             const float *data, float lambda_feature,
                                             int64_t feature_warmup_epochs, int *has_empty_row);
/* The rejections of a feature-aware epoch (:759-761 "Feature-aware iALS does not support IALSPP.",
 * the weight shape of :1016-1042, the empty-row guard of :639-652 with the given OR over all
 * ranks), from state that is the same on every rank: a caller that runs it before the epoch's
 * first collective sees every rank fail alike, before any factor or weight changes. */
IALS_API int ials_trainer_check_shard_step(ials_trainer *t, const ials_solver_config *solver,
                                           int user_has_empty_row, int item_has_empty_row);
/* The rank's partial sums of the weight refit W = (F^T D F + lambda I)^-1 F^T D X
 * (initialize_feature_weight_cache :1083-1132, solve_feature_weight :1134-1180) over its own rows,
 * D = diag(compute_reg) of those rows: F^T D F in a trainer-owned device buffer of n_w * n_w floats
 * (only before the first refit: the factor is cached, like cache_ready; count 0 afterwards) and
 * F^T D X in one of n_w * ld floats.  Both counts are 0 when the side's last solve used no prior.
 * The caller all-reduces (sum) each buffer in place. */
IALS_API int ials_trainer_feature_partials(ials_trainer *t, int side, float **d_gram, int64_t *gram_count,
                                           float **d_rhs, int64_t *rhs_count);
/* After that all-reduce: factors F^T D F + lambda I (first time only), solves for W and stores it
 * as the side's weight.  No-op when ials_trainer_feature_partials returned zero counts.
 * "Feature ridge Cholesky decomposition failed." / "Feature ridge solve failed." surface at the
 * next ials_trainer_sync. */
IALS_API int ials_trainer_feature_refit(ials_trainer *t, int side);
/* This rank's share of IALSTrainer::compute_loss (:836-940), halved, in float64: the data term and
 * the regulariser (|x - prior|^2 for a side with features) of its own user rows and the
 * regulariser of its own item rows; with include_global != 0 also sum(P_user .* P_item) / alpha0
 * from the full replicas and lambda |W|^2 of each side with features.  The sum over ranks, with
 * include_global on exactly one of them, is the loss.  Reads the full replicas: every rank's
 * solves must have completed (ials_trainer_sync + a barrier). */
IALS_API int ials_trainer_compute_loss_shard(ials_trainer *t, const ials_solver_config *solver, int include_global,
                                             double *out);
/* CUDA IPC plumbing for peer replicas: 64-byte handle of this trainer's factor
 * matrix; registration of the peers' handles (world entries, own rank skipped). */
IALS_API int ials_trainer_ipc_handle(ials_trainer *t, int side, unsigned char handle_out[64]);
IALS_API int ials_trainer_ipc_open_peers(ials_trainer *t, int side, const unsigned char *handles,
                                int world, int rank);

#ifdef __cplusplus
}
#endif
#endif /* IALS_B200_H */
