// The trainer object behind the C ABI (include/ials_b200.h) and the host helpers shared by the
// api*.cu / solve.cu translation units (internal).
#pragma once
#include <functional>
#include <memory>
#include <string>
#include <vector>

#include "common.cuh"

struct ials_trainer {
  ials_model_config cfg{};
  int device = 0;
  cudaStream_t stream = nullptr;
  int64_t U = 0, I = 0;
  int K = 0, ld = 0;
  ials::DeviceBuffer<float> factor[2];  // [0] user U x ld, [1] item I x ld
  ials::DeviceCsr X, Xt;
  bool has_X = false;
  ials::DeviceBuffer<float> P[2];  // P[0]: user_solver.P = alpha0 item^T item; P[1]: item_solver.P
  ials::DeviceBuffer<float> gram_scratch;
  ials::GramWorkspace gws;  // tensor-core Gram (ld == 128)
  // heavy-row path of the CG solver: per-job Gram partials from wgram.cu (grow-only)
  ials::DeviceBuffer<float> heavy_W, heavy_b;
  ials::DeviceBuffer<int> err_flags;
  ials::DeviceBuffer<unsigned long long> work_counter;
  ials::DeviceBuffer<double> d_loss;
  ials::DeviceBuffer<unsigned char> score_buf;
  // ials_trainer_recommend: result and mask staging buffers, kept between calls (grow-only) --
  // an Evaluator calls it once per block of users, and five cudaMalloc / cudaFree pairs per call
  // cost as much as the kernel itself at 128 .. 4096 users per block
  ials::DeviceBuffer<int32_t> rec_idx, rec_count, rec_mindices, rec_aindices;
  ials::DeviceBuffer<int64_t> rec_mindptr, rec_aindptr, rec_uidx;
  ials::DeviceBuffer<float> rec_score, rec_users, rec_emb;
  std::vector<uint32_t> rec_abitmap_host;  // shared allow-list as a bitmap, staged for the upload
  // ials_trainer_similar (grow-only): the side's rows scaled to unit norm, and the mask CSR whose row i
  // hides row i (the query itself, for a range of queries without forbidden lists)
  ials::DeviceBuffer<float> sim_norm;
  ials::DeviceBuffer<int64_t> sim_self_indptr;
  ials::DeviceBuffer<int32_t> sim_self_indices;
  // candidate ranking (grow-only): the first score task of each query row (launch_cand_scores)
  ials::DeviceBuffer<int64_t> cand_tasks;
  // explanations (grow-only): the schedule, slot -> pair and pair -> contribution offsets, targets, cold
  // rows, and per slab the pair scores / priors and the contribution scratch; host copies of the indptr
  // of X and Xt, made on first use (the training matrices never change)
  ials::DeviceBuffer<int64_t> expl_offsets, expl_hist_indptr;
  ials::DeviceBuffer<int32_t> expl_rows, expl_targets, expl_hist_indices, expl_contrib_idx;
  ials::DeviceBuffer<float> expl_hist_data, expl_pair_out, expl_contrib;
  std::vector<int64_t> indptr_host[2];
  // shard (multi-GPU): rows owned (solved) by this rank, per side; X / Xt then hold only
  // those rows (DeviceCsr::row_base = shard begin) while both factor matrices are full replicas
  bool sharded = false;
  int64_t shard[2][2] = {{0, 0}, {0, 0}};
  int n_peers[2] = {0, 0};
  float *peers[2][8] = {};
  // phase timing: 5 events per profiled epoch (before, after each of the 4 phases)
  bool profiling = false;
  std::vector<cudaEvent_t> prof_events;
  // ials_trainer_step_io: second stream + event for the overlapped read-back of the user factors
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t users_done = nullptr;
  ials::DeviceBuffer<int> ready_flags;  // step_io: one flag per chunk of user rows arriving from the host
  ials::PinnedBuffer<int> ready_host;   // pinned source of the flag copies
  ials::DeviceBuffer<int32_t> order_io; // step_io: the light user rows by (arrival chunk, descending degree)
  int ready_token = 0;
  bool ready_pending = false;          // a flagged upload is in flight for the next user solve
  cudaEvent_t upload_done = nullptr;   // behind its last chunk, on the copy stream
  // Routes that form the normal equations of every row on the tensor cores (256-column Cholesky,
  // iALS++): a job plan over EVERY non-empty row of X / Xt, built on first use, the host copy of
  // its row -> job map (empty: not built yet), and the per-chunk workspaces of Gram blocks
  ials::JobPlan all_rows[2];
  std::vector<int32_t> all_rows_first[2];
  ials::DeviceBuffer<float> chol_ws;  // jobs per chunk x (W [256][256] | b [kWGram256BParts][256])
  ials::DeviceBuffer<float> gs_ws;    // iALS++ route: W [jobs][128][128] | b [jobs][kWGramBParts][128]
  ials::DeviceBuffer<unsigned char> chol_scratch;  // cholesky_ll_kernel: the factor of every resident CTA
  // feature-aware iALS (IALSTrainer(config, X, user_feature, item_feature), IALSTrainer.hpp:722-743)
  struct FeatureSide {
    bool given = false;       // the trainer was built with features for this side
    bool weight_set = false;  // a weight matrix exists (given, or restored by set_feature_weight)
    bool has_empty_row = false;
    ials::FeatureDev F;       // views of the owned device arrays below
    ials::DeviceBuffer<float> dense;
    ials::DeviceCsr csr;
    int64_t n_w = 0;                   // rows of the weight (= feature columns)
    ials::DeviceBuffer<float> weight;  // [n_w x ld]
    ials::DeviceBuffer<float> prior;   // [F.n_rows x ld] (a row-sharded trainer: its own rows only)
    ials::DeviceBuffer<float> rw;      // [n_rows]   compute_reg of every row (FeatureWeightCache::row_weights)
    ials::DeviceBuffer<float> llt;     // [n_w x n_w] Cholesky factor of F^T D F + lambda I (FeatureWeightCache::llt)
    ials::DeviceBuffer<float> rhs;     // [n_w x ld]
    bool cache_ready = false;
    // row-sharded trainer: the last ials_trainer_solve_shard of this side used the prior, so its
    // weight refit (ials_trainer_feature_partials / _feature_refit) is due
    bool refit_pending = false;
    float lambda = 0.f;
  } feat[2];
  bool feature_aware = false;
  int64_t epoch = 0, feature_warmup = 0;  // epoch_, config_.feature_warmup_epochs
  int64_t n_rows(int side) const { return side == 0 ? U : I; }
};

namespace ials {

extern thread_local std::string g_last_error;

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    CUDA_CHECK(cudaGetDevice(&prev));
    if (prev != dev) CUDA_CHECK(cudaSetDevice(dev));
    else prev = -1;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

template <typename F>
int guarded(F &&fn) {
  try {
    fn();
    return IALS_OK;
  } catch (const InvalidArgument &e) {
    g_last_error = e.what();
    return IALS_ERR_INVALID_ARGUMENT;
  } catch (const NotImplemented &e) {
    g_last_error = e.what();
    return IALS_ERR_NOT_IMPLEMENTED;
  } catch (const CudaError &e) {
    g_last_error = e.what();
    cudaGetLastError();  // clear the sticky-less error state
    return IALS_ERR_CUDA;
  } catch (const std::invalid_argument &e) {
    g_last_error = e.what();
    return IALS_ERR_INVALID_ARGUMENT;
  } catch (const std::exception &e) {
    g_last_error = e.what();
    return IALS_ERR_RUNTIME;
  } catch (...) {  // nothing may unwind through the C ABI
    g_last_error = "unknown C++ exception";
    return IALS_ERR_RUNTIME;
  }
}

inline void require(bool cond, const char *msg) {
  if (!cond) throw InvalidArgument(msg);
}

inline void require_side(int side) { require(side == 0 || side == 1, "side must be 0 or 1"); }

// Padded row copies: host rows of K floats <-> device rows of ld floats, synchronous or on stream s
inline void rows_to_device(float *dst, int64_t ld, const float *src, int64_t K, int64_t n) {
  CUDA_CHECK(cudaMemcpy2D(dst, sizeof(float) * ld, src, sizeof(float) * K, sizeof(float) * K, n,
                          cudaMemcpyHostToDevice));
}
inline void rows_to_device(float *dst, int64_t ld, const float *src, int64_t K, int64_t n, cudaStream_t s) {
  CUDA_CHECK(cudaMemcpy2DAsync(dst, sizeof(float) * ld, src, sizeof(float) * K, sizeof(float) * K, n,
                               cudaMemcpyHostToDevice, s));
}
inline void rows_to_host(float *dst, int64_t K, const float *src, int64_t ld, int64_t n) {
  CUDA_CHECK(cudaMemcpy2D(dst, sizeof(float) * K, src, sizeof(float) * ld, sizeof(float) * K, n,
                          cudaMemcpyDeviceToHost));
}
inline void rows_to_host(float *dst, int64_t K, const float *src, int64_t ld, int64_t n, cudaStream_t s) {
  CUDA_CHECK(cudaMemcpy2DAsync(dst, sizeof(float) * K, src, sizeof(float) * ld, sizeof(float) * K, n,
                               cudaMemcpyDeviceToHost, s));
}

// Phase marks are per epoch (ials_trainer_step*) only: a scope that solves outside an epoch turns them off
struct NoProfiling {
  ials_trainer *t;
  bool saved;
  explicit NoProfiling(ials_trainer *t_) : t(t_), saved(t_->profiling) { t->profiling = false; }
  ~NoProfiling() { t->profiling = saved; }
};

// A trainer under construction: a failed create* releases it through ials_trainer_destroy
using TrainerPtr = std::unique_ptr<ials_trainer, void (*)(ials_trainer *)>;

// api.cu
void require_device(int device);
void check_solver(const ials_solver_config *sc);
void alloc_common(ials_trainer *t);
TrainerPtr new_trainer(const ials_model_config *cfg, int64_t U, int64_t I, int device);
void init_factors(ials_trainer *t, bool on_device);
int64_t env_int(const char *name, int64_t dflt);
int64_t heavy_job_len();  // IALS_HEAVY_JOB_LEN (default 4096); anything but a positive integer is rejected
void plan_csr(ials_trainer *t, DeviceCsr &csr);
void copy_csr(DeviceCsr &d, int64_t n_rows, int64_t n_cols, int64_t nnz, const int64_t *indptr,
              const int32_t *indices, const float *data, cudaMemcpyKind kind);
void upload_csr(DeviceCsr &d, int64_t n_rows, int64_t n_cols, const int64_t *indptr,
                const int32_t *indices, const float *data, bool on_device = false);
void gram_rows(ials_trainer *t, int src, int64_t begin, int64_t end, float *dst);
void prof_mark(ials_trainer *t);
void gram_side(ials_trainer *t, int solver_side);
void sync_and_check(ials_trainer *t);
void fold_in(ials_trainer *t, int side, int64_t n_rows, int64_t n_cols, const int64_t *indptr,
             const int32_t *indices, const float *data, const ials_solver_config *solver, float *out_host,
             const std::function<const float *(const DeviceCsr &)> &stage_prior = nullptr);
// solve.cu
SolveArgs make_args(ials_trainer *t, int side, float *target, const DeviceCsr &csr,
                    const ials_solver_config *sc);
void run_solver(ials_trainer *t, const SolveArgs &a, const DeviceCsr &csr,
                const ials_solver_config *sc, cudaStream_t s);
void ensure_copy_stream(ials_trainer *t);
void enqueue_flagged_user_upload(ials_trainer *t, int64_t row_begin, int64_t n_rows, const float *rows_host);
void consume_flagged_upload(ials_trainer *t, const ials_solver_config *sc, SolveArgs &a, int64_t row_begin);
// api_recommend.cu: top-k lists of `rows` query rows against a catalogue, everything already on the
// device (the recommend entry points and the evaluation sets: user rows against the item factors;
// ials_trainer_similar: rows of one side against that side).  The fused
// tensor-core kernel where it applies (score_topk_tc_supported, sorted mask rows), else scores + mask +
// SIMT top-k; allow-lists and users picked by index with mask_mode 0 need the fused route
// (NotImplemented otherwise).  Enqueued on t->stream.
constexpr int64_t kListSlabRows = 262144;  // rows per fused launch: bounds its scratch (score_buf)
struct ListJob {
  const float *user_rows = nullptr;  // [rows x ld] queries
  const float *catalog = nullptr;    // [n_catalog x ld] rows ranked for each query
  int64_t n_catalog = 0;
  int64_t rows = 0, k = 0;
  int mask_mode = 1;                 // 0: rows of X, 1: none, 2: the CSR below
  int64_t x_row0 = 0;                // mode 0: row of X (local to the shard) that masks block row 0
  const int64_t *rowmap = nullptr;   // mode 0, users picked by index: block row r is user rowmap[r]
  const int64_t *m_indptr = nullptr; // mode 2: block row r is masked by CSR row m_row0 + r
  const int32_t *m_indices = nullptr;
  int64_t m_row0 = 0;
  bool mask_sorted = true;           // column ids strictly ascending in every mask row
  int64_t allow_n_lists = 0;         // 0, 1 (a_bitmap) or per row (CSR row a_row0 + r)
  const int64_t *a_indptr = nullptr;
  const int32_t *a_indices = nullptr;
  const uint32_t *a_bitmap = nullptr;
  int64_t a_row0 = 0;
  int32_t *idx = nullptr;            // [rows x k] out
  float *score = nullptr;            // [rows x k] out
  int32_t *count = nullptr;          // [rows] out
};
void produce_lists(ials_trainer *t, const ListJob &j);
// Validates a host mask CSR of `rows` rows over n_cols items and copies it into d_indptr / d_indices
// (grown as needed) on stream s
void stage_mask(int64_t rows, int64_t n_cols, const int64_t *indptr, const int32_t *indices,
                DeviceBuffer<int64_t> &d_indptr, DeviceBuffer<int32_t> &d_indices, cudaStream_t s);
bool mask_rows_sorted(int64_t rows, const int64_t *indptr, const int32_t *indices);
// Validates host allow-lists (strictly ascending int32 ids in [0, n_items)) and uploads them on stream s
// into job.allow_n_lists / a_bitmap (one shared list, staged in `words`) or a_indptr / a_indices
void stage_allow_lists(int64_t n_items, int64_t n_lists, const int64_t *indptr, const int32_t *indices,
                       std::vector<uint32_t> &words, DeviceBuffer<int64_t> &d_indptr,
                       DeviceBuffer<int32_t> &d_indices, cudaStream_t s, ListJob &job);
// api_features.cu
void check_prior_defined(const ials_trainer *t, int side, bool has_empty_row);
bool side_uses_features(const ials_trainer *t, int side);
void check_feature_weight_shapes(const ials_trainer *t, bool any_epoch);
const float *stored_prior(ials_trainer *t, int side);
void update_feature_weight(ials_trainer *t, int side);
void check_feature_solver(const ials_trainer *t, const ials_solver_config *sc);

}  // namespace ials
