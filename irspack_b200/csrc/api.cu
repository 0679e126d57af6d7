// C ABI of libials_b200.so (include/ials_b200.h): the trainer object that
// replaces irspack's `_ials_core.IALSTrainer`
// (/root/reference/cpp_source/als/IALSTrainer.hpp:709-984, wrapper.cpp:130-181).
#include <algorithm>
#include <cerrno>
#include <cmath>
#include <cstdlib>
#include <random>
#include <string>
#include <vector>

#include "trainer.cuh"

using namespace ials;

namespace ials {

int64_t g_kernel_launches = 0;
thread_local std::string g_last_error;

void require_device(int device) {
  int n_dev = 0;
  if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) {
    cudaGetLastError();
    throw CudaError("no CUDA device available: the B200 backend has no CPU fallback");
  }
  require(device >= 0 && device < n_dev, "invalid CUDA device index");
}

void check_solver(const ials_solver_config *sc) {
  require(sc != nullptr, "solver_config is null");
  // Solver::prepare_p, IALSTrainer.hpp:81-83
  require(sc->n_threads > 0, "n_threads must be strictly positive.");
  require(sc->solver_type == IALS_SOLVER_CG || sc->solver_type == IALS_SOLVER_CHOLESKY ||
              sc->solver_type == IALS_SOLVER_IALSPP,
          "unknown solver_type");
  require(sc->max_cg_steps >= 0, "max_cg_steps must be non-negative");
  if (sc->solver_type == IALS_SOLVER_IALSPP) {
    // the reference's block loop never ends with a zero step (IALSTrainer.hpp:526-527)
    require(sc->ialspp_subspace_dimension >= 1, "ialspp_subspace_dimension must be strictly positive.");
    require(sc->ialspp_iteration >= 0, "ialspp_iteration must be non-negative");
  }
}

void alloc_common(ials_trainer *t) {
  const int64_t ld = t->ld;
  for (int side = 0; side < 2; side++) {
    const int64_t n = t->n_rows(side);
    CUDA_CHECK(cudaMemset(t->factor[side].alloc(std::max<int64_t>(n * ld, 1)), 0,
                          sizeof(float) * std::max<int64_t>(n * ld, 1)));
    CUDA_CHECK(cudaMemset(t->P[side].alloc(ld * ld), 0, sizeof(float) * ld * ld));
  }
  t->gram_scratch.alloc(ld * ld);
  if (ld == 128) t->gws.alloc(kNumSMsB200);
  CUDA_CHECK(cudaMemset(t->err_flags.alloc(kNumErrFlags), 0, sizeof(int) * kNumErrFlags));
  t->work_counter.alloc(1);
  t->d_loss.alloc(1);
}

// Validates the model and the device; the trainer holds no device memory yet.  Its deleter is
// ials_trainer_destroy, which frees on the trainer's device after a synchronise.
TrainerPtr new_trainer(const ials_model_config *cfg, int64_t U, int64_t I, int device) {
  require(cfg != nullptr, "model_config is null");
  require(cfg->K >= 1 && cfg->K <= 512, "K must be in [1, 512]");
  require(U >= 0 && I >= 0, "negative matrix shape");
  require(U < (1ll << 31) && I < (1ll << 31), "matrix dimensions must fit int32");
  require(cfg->loss_type == IALS_LOSS_ORIGINAL || cfg->loss_type == IALS_LOSS_IALSPP,
          "unknown loss_type");
  require_device(device);
  TrainerPtr t(new ials_trainer(), ials_trainer_destroy);
  t->cfg = *cfg;
  t->device = device;
  t->U = U;
  t->I = I;
  t->K = (int)cfg->K;
  // Row stride of the factor matrices.  Every K <= 128 is padded to 128 floats (zero columns
  // that stay zero): the tuned kernels (tcgen05 Gram, cg_rows, dense CG, fused scoring) are
  // written for 512-byte rows, and even at K = 64 they beat the generic-K kernels 3x
  // (ML-1M shape: 1.64 vs 5.13 ms/epoch, profiles/r01l_c1_final.json, r01k_c1.json).
  t->ld = cfg->K <= 128 ? 128 : (int)round_up(cfg->K, 32);
  return t;
}

// Solver::initialize, IALSTrainer.hpp:64-76: a fresh mt19937(seed) per matrix; on_device: the
// counter-based device fill (for factor matrices too large for the serial host RNG)
void init_factors(ials_trainer *t, bool on_device) {
  if (!(t->cfg.init_stdev > 0)) return;  // matrices stay zero
  if (on_device) {
    const float sd = (float)(t->cfg.init_stdev / std::sqrt((double)t->K));
    // same seed for both matrices, like the reference's two fresh generators
    for (int side = 0; side < 2; side++)
      launch_init_normal(t->factor[side].get(), t->n_rows(side), t->K, t->ld, sd,
                         (uint64_t)(uint32_t)t->cfg.random_seed, t->stream);
    CUDA_CHECK(cudaStreamSynchronize(t->stream));
    return;
  }
  for (int side = 0; side < 2; side++) {
    const int64_t n = t->n_rows(side);
    if (n == 0) continue;
    std::mt19937 gen(t->cfg.random_seed);
    std::normal_distribution<float> dist(0.0, t->cfg.init_stdev / std::sqrt((double)t->K));
    std::vector<float> h((size_t)n * t->K);
    for (auto &v : h) v = dist(gen);
    rows_to_device(t->factor[side].get(), t->ld, h.data(), t->K, n);
  }
}

// Schedule of a CSR side (K padded to 128).  Rows are sorted by descending degree and cut into
// two classes:
//   degree > IALS_HEAVY_THRESHOLD (default 2048): "heavy" -- tensor-core Gram of the gathered
//     neighbours + dense CG; their neighbour lists are cut into jobs of <= IALS_HEAVY_JOB_LEN
//     (default 4096) entries;
//   the rest: "light" -- warp-per-row batches (cg_rows.cu).
// Rows of a matrix with a negative stored value all take the light path (the sqrt-weighted
// Gram does not exist then).  The two knobs exist because the best cut depends on where the
// gathered matrix lives: 2048 when it is L2-resident (ML-20M shape, r01g / r02a sweeps); lower
// when it streams from HBM and the four passes of the light path cost four reads (configs[3]).
int64_t env_int(const char *name, int64_t dflt) {
  const char *e = std::getenv(name);
  return e != nullptr && *e ? std::atoll(e) : dflt;
}
// A job length of 0 would divide by zero when the plan cuts a row, and a negative one never ends it.
int64_t heavy_job_len() {
  const char *e = std::getenv("IALS_HEAVY_JOB_LEN");
  if (e == nullptr || !*e) return 4096;
  char *end = nullptr;
  errno = 0;
  const long long v = std::strtoll(e, &end, 10);
  require(*end == '\0' && errno == 0 && v >= 1, "IALS_HEAVY_JOB_LEN must be a positive integer");
  return v;
}
void plan_csr(ials_trainer *t, DeviceCsr &csr) {
  build_row_order(csr, t->stream);
  csr.has_negative = csr_has_negative(csr, t->stream);
  if (t->ld == 128) {
    const int64_t heavy = std::max<int64_t>(env_int("IALS_HEAVY_THRESHOLD", 2048), 1);
    build_heavy_plan(csr, heavy, heavy_job_len(), csr.heavy, t->stream);
  }
}

// Copies a CSR (host or device arrays) into device memory owned by `d`.
void upload_csr(DeviceCsr &d, int64_t n_rows, int64_t n_cols, const int64_t *indptr,
                const int32_t *indices, const float *data, bool on_device) {
  require(indptr != nullptr, "indptr is null");
  int64_t nnz = 0;
  if (on_device) {
    CUDA_CHECK(cudaMemcpy(&nnz, indptr + n_rows, sizeof(int64_t), cudaMemcpyDeviceToHost));
    require(nnz >= 0, "bad indptr");
  } else {
    require(indptr[0] == 0, "indptr[0] must be 0");
    for (int64_t r = 0; r < n_rows; r++) require(indptr[r + 1] >= indptr[r], "indptr must be non-decreasing");
    nnz = indptr[n_rows];
  }
  require(nnz <= kMaxGramEntries,
          "nnz must be at most 2^31 - 64 (int32 offsets, as in the reference's Eigen StorageIndex, with room for "
          "the tensor-core Gram's last pipeline stage)");
  require(nnz == 0 || (indices != nullptr && data != nullptr), "indices/data are null");
  if (!on_device)
    for (int64_t j = 0; j < nnz; j++)
      require(indices[j] >= 0 && indices[j] < n_cols, "column index out of range");
  copy_csr(d, n_rows, n_cols, nnz, indptr, indices, data,
           on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice);
}

// Copies the arrays of a validated CSR into device memory owned by `d`.
void copy_csr(DeviceCsr &d, int64_t n_rows, int64_t n_cols, int64_t nnz, const int64_t *indptr,
              const int32_t *indices, const float *data, cudaMemcpyKind kind) {
  d.n_rows = n_rows;
  d.n_cols = n_cols;
  d.nnz = nnz;
  d.indptr.alloc(n_rows + 1);
  d.indices.alloc(std::max<int64_t>(nnz, 1));
  d.data.alloc(std::max<int64_t>(nnz, 1));
  CUDA_CHECK(cudaMemcpy(d.indptr.get(), indptr, sizeof(int64_t) * (n_rows + 1), kind));
  if (nnz) {
    CUDA_CHECK(cudaMemcpy(d.indices.get(), indices, sizeof(int32_t) * nnz, kind));
    CUDA_CHECK(cudaMemcpy(d.data.get(), data, sizeof(float) * nnz, kind));
  }
}

// tcgen05 Gram when the row stride is 128, FP32 SIMT (gram.cu) for the other ranks
bool gram_use_tensor_cores(const ials_trainer *t) { return t->ld == 128 && t->gws.max_jobs > 0; }

void gram_rows(ials_trainer *t, int src, int64_t begin, int64_t end, float *dst) {
  if (gram_use_tensor_cores(t))
    launch_gram_tc(t->factor[src].get(), begin, end, t->cfg.alpha0, t->gws, dst, t->stream);
  else
    launch_gram(t->factor[src].get(), begin, end, t->ld, t->cfg.alpha0, t->gram_scratch.get(), dst, t->stream);
}

// Phase timing: one event per mark; an epoch records kMarksPerEpoch marks
//   start | Gram(item) | users: wgram, dense CG, light rows | Gram(user) | items: wgram, dense, light
constexpr int kMarksPerEpoch = 9;
void prof_mark(ials_trainer *t) {
  if (!t->profiling) return;
  cudaEvent_t e;
  CUDA_CHECK(cudaEventCreate(&e));
  t->prof_events.push_back(e);
  CUDA_CHECK(cudaEventRecord(e, t->stream));
}

void gram_side(ials_trainer *t, int solver_side) {
  // solver_side 0 (users) needs alpha0 * item^T item, and vice versa
  const int src = 1 - solver_side;
  gram_rows(t, src, 0, t->n_rows(src), t->P[solver_side].get());
}

void sync_and_check(ials_trainer *t) {
  if (t->ready_pending && t->copy_stream) CUDA_CHECK(cudaStreamSynchronize(t->copy_stream));  // an upload nobody consumed
  int flags[kNumErrFlags];
  CUDA_CHECK(cudaMemcpyAsync(flags, t->err_flags.get(), sizeof(flags), cudaMemcpyDeviceToHost, t->stream));
  CUDA_CHECK(cudaStreamSynchronize(t->stream));
  if (flags[kErrCgSingular] || flags[kErrCholDecomp] || flags[kErrCholSolve] || flags[kErrInternal] ||
      flags[kErrFeatureLlt] || flags[kErrFeatureSolve]) {
    CUDA_CHECK(cudaMemsetAsync(t->err_flags.get(), 0, sizeof(flags), t->stream));
    // messages of IALSTrainer.hpp:252-253, 318, 322
    if (flags[kErrInternal]) throw std::runtime_error("internal error: a row was scheduled on a kernel that cannot hold it");
    if (flags[kErrFeatureLlt]) throw std::runtime_error("Feature ridge Cholesky decomposition failed.");  // :1107
    if (flags[kErrFeatureSolve]) throw std::runtime_error("Feature ridge solve failed.");                  // :1171
    if (flags[kErrCgSingular]) throw std::runtime_error("Conjugate-gradient solver encountered a singular system.");
    if (flags[kErrCholDecomp]) throw std::runtime_error("Cholesky decomposition failed.");
    throw std::runtime_error("Cholesky solve failed.");
  }
}

// Fold-in (Solver::X_to_vector, IALSTrainer.hpp:123-140, :791-801): solves the rows of the host CSR
// (side 0) or of its transpose (side 1) against the trainer's other factor matrix, starting from zero.
// stage_prior (X_to_vector_with_prior, :142-167) is given the planned CSR of the new rows and returns
// device rows [n_new x ld] that the solve starts from and is regularised towards.
void fold_in(ials_trainer *t, int side, int64_t n_rows, int64_t n_cols, const int64_t *indptr,
             const int32_t *indices, const float *data, const ials_solver_config *solver, float *out_host,
             const std::function<const float *(const DeviceCsr &)> &stage_prior) {
  DeviceCsr given, transposed;
  DeviceBuffer<float> target;
  StreamSyncOnExit sync{t->stream};
  upload_csr(given, n_rows, n_cols, indptr, indices, data);
  if (side == 1) build_transpose(given, transposed, t->stream);  // X.transpose(), :800
  DeviceCsr &csr = side == 1 ? transposed : given;
  plan_csr(t, csr);
  const int64_t n_new = csr.n_rows;
  const float *prior = stage_prior ? stage_prior(csr) : nullptr;
  const size_t bytes = sizeof(float) * std::max<int64_t>(n_new * t->ld, 1);
  target.alloc(std::max<int64_t>(n_new * t->ld, 1));
  if (prior)
    CUDA_CHECK(cudaMemcpyAsync(target.get(), prior, bytes, cudaMemcpyDeviceToDevice, t->stream));  // result = prior, :156
  else
    CUDA_CHECK(cudaMemsetAsync(target.get(), 0, bytes, t->stream));  // DenseMatrix::Zero, :132
  gram_side(t, side);  // prepare_p, :793 / :799
  SolveArgs a = make_args(t, side, target.get(), csr, solver);
  a.prior = prior;
  run_solver(t, a, csr, solver, t->stream);
  if (n_new) {
    require(out_host != nullptr, "out is null");
    rows_to_host(out_host, t->K, target.get(), t->ld, n_new, t->stream);
  }
  sync_and_check(t);
}

}  // namespace ials

namespace {

void finish_csr(ials_trainer *t) {
  build_transpose(t->X, t->Xt, t->stream);
  plan_csr(t, t->X);
  plan_csr(t, t->Xt);
  t->has_X = true;
}

// One half-epoch of IALSTrainer::step (:758-789) on the trainer's own matrices: Gram, solve
// (with the stored feature prior once the warm-up epochs are over), feature-weight update.
void epoch_side(ials_trainer *t, int side, const ials_solver_config *sc, SolveArgs *io_args = nullptr) {
  gram_side(t, side);
  prof_mark(t);
  const DeviceCsr &csr = side == 0 ? t->X : t->Xt;
  SolveArgs a = io_args ? *io_args : make_args(t, side, t->factor[side].get(), csr, sc);
  const bool with_features = side_uses_features(t, side);
  if (with_features) {
    check_prior_defined(t, side, t->feat[side].has_empty_row);
    a.prior = stored_prior(t, side);
  }
  run_solver(t, a, csr, sc, t->stream);  // records three marks
  if (with_features) update_feature_weight(t, side);
}

void half_step(ials_trainer *t, int side, const ials_solver_config *sc) {
  NoProfiling guard(t);
  if (t->sharded) throw std::runtime_error("sharded trainer: drive the epoch with gram_partial / solve_shard");
  if (!t->has_X) throw std::runtime_error("this trainer was restored without its interaction matrix; it cannot train");
  check_feature_solver(t, sc);
  check_feature_weight_shapes(t, false);
  epoch_side(t, side, sc);  // (a test entry: the epoch counter is not advanced)
}

}  // namespace

extern "C" {

const char *ials_last_error(void) { return g_last_error.c_str(); }
const char *ials_version(void) { return "0.1.0"; }
int ials_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int ials_trainer_create(const ials_model_config *config, int64_t n_users, int64_t n_items,
                        const int64_t *indptr, const int32_t *indices, const float *data,
                        int device, ials_trainer **out) {
  return guarded([&] {
    require(out != nullptr, "out is null");
    *out = nullptr;
    TrainerPtr t = new_trainer(config, n_users, n_items, device);
    DeviceGuard g(device);
    alloc_common(t.get());
    upload_csr(t->X, n_users, n_items, indptr, indices, data);
    finish_csr(t.get());
    init_factors(t.get(), false);
    *out = t.release();
  });
}

int ials_trainer_create_from_device_csr(const ials_model_config *config, int64_t n_users,
                                        int64_t n_items, const int64_t *d_indptr,
                                        const int32_t *d_indices, const float *d_data, int device,
                                        int init_on_device, ials_trainer **out) {
  return guarded([&] {
    require(out != nullptr, "out is null");
    *out = nullptr;
    TrainerPtr t = new_trainer(config, n_users, n_items, device);
    DeviceGuard g(device);
    alloc_common(t.get());
    upload_csr(t->X, n_users, n_items, d_indptr, d_indices, d_data, /*on_device=*/true);
    finish_csr(t.get());
    init_factors(t.get(), init_on_device != 0);
    *out = t.release();
  });
}

int ials_trainer_create_from_factors(const ials_model_config *config, int64_t n_users,
                                     int64_t n_items, const float *user, const float *item,
                                     int device, ials_trainer **out) {
  return guarded([&] {
    require(out != nullptr, "out is null");
    *out = nullptr;
    TrainerPtr t = new_trainer(config, n_users, n_items, device);
    DeviceGuard g(device);
    alloc_common(t.get());
    require((n_users == 0 || user) && (n_items == 0 || item), "factor pointer is null");
    const float *src[2] = {user, item};
    for (int side = 0; side < 2; side++)
      if (t->n_rows(side)) rows_to_device(t->factor[side].get(), t->ld, src[side], t->K, t->n_rows(side));
    // the reference rebuilds both P matrices on unpickle (IALSTrainer.hpp:751-755)
    gram_side(t.get(), 0);
    gram_side(t.get(), 1);
    CUDA_CHECK(cudaStreamSynchronize(t->stream));
    *out = t.release();
  });
}

void ials_trainer_destroy(ials_trainer *t) {
  if (!t) return;
  int prev = -1;
  cudaGetDevice(&prev);
  cudaSetDevice(t->device);
  cudaDeviceSynchronize();
  for (int side = 0; side < 2; side++)
    for (int p = 0; p < t->n_peers[side]; p++)
      if (t->peers[side][p]) cudaIpcCloseMemHandle(t->peers[side][p]);
  for (auto e : t->prof_events) cudaEventDestroy(e);
  if (t->users_done) cudaEventDestroy(t->users_done);
  if (t->upload_done) cudaEventDestroy(t->upload_done);
  if (t->copy_stream) cudaStreamDestroy(t->copy_stream);
  delete t;  // the buffers free themselves, with the trainer's device current
  cudaGetLastError();
  if (prev >= 0) cudaSetDevice(prev);
}

int ials_trainer_set_stream(ials_trainer *t, void *cuda_stream) {
  return guarded([&] {
    require(t != nullptr, "trainer is null");
    t->stream = (cudaStream_t)cuda_stream;
  });
}

int ials_trainer_step_async(ials_trainer *t, const ials_solver_config *solver) {
  return guarded([&] {
    require(t != nullptr, "trainer is null");
    check_solver(solver);
    if (t->sharded) throw std::runtime_error("sharded trainer: drive the epoch with gram_partial / solve_shard");
    DeviceGuard g(t->device);
    if (!t->has_X) throw std::runtime_error("this trainer was restored without its interaction matrix; it cannot train");
    check_feature_solver(t, solver);
    check_feature_weight_shapes(t, false);
    prof_mark(t);
    for (int side = 0; side < 2; side++) epoch_side(t, side, solver);  // IALSTrainer.hpp:762-787
    t->epoch++;
  });
}

int ials_trainer_set_profiling(ials_trainer *t, int enabled) {
  return guarded([&] {
    require(t != nullptr, "trainer is null");
    t->profiling = enabled != 0;
  });
}

int ials_trainer_get_timings(ials_trainer *t, double ms[8], int64_t *n_epochs) {
  return guarded([&] {
    require(t != nullptr && ms != nullptr && n_epochs != nullptr, "null argument");
    DeviceGuard g(t->device);
    CUDA_CHECK(cudaStreamSynchronize(t->stream));
    for (int i = 0; i < kMarksPerEpoch - 1; i++) ms[i] = 0.0;
    *n_epochs = (int64_t)t->prof_events.size() / kMarksPerEpoch;
    for (size_t b = 0; b + kMarksPerEpoch <= t->prof_events.size(); b += kMarksPerEpoch) {
      for (int i = 0; i < kMarksPerEpoch - 1; i++) {
        float v = 0.f;
        CUDA_CHECK(cudaEventElapsedTime(&v, t->prof_events[b + i], t->prof_events[b + i + 1]));
        ms[i] += v;
      }
    }
    for (auto e : t->prof_events) cudaEventDestroy(e);
    t->prof_events.clear();
  });
}

int ials_trainer_plan_stats(ials_trainer *t, int side, int64_t out[8]) {
  return guarded([&] {
    require(t != nullptr && out != nullptr, "null argument");
    require_side(side);
    const DeviceCsr &c = side == 0 ? t->X : t->Xt;
    out[0] = c.n_rows;
    out[1] = c.nnz;
    out[2] = c.heavy.n_heavy;
    out[3] = c.heavy.nnz_heavy;
    out[4] = c.heavy.n_jobs;
    out[5] = c.max_degree;
    out[6] = c.has_negative ? 1 : 0;
    out[7] = 0;
  });
}

int64_t ials_kernel_launch_count(void) { return __atomic_load_n(&ials::g_kernel_launches, __ATOMIC_RELAXED); }

int ials_trainer_sync(ials_trainer *t) {
  return guarded([&] {
    require(t != nullptr, "trainer is null");
    DeviceGuard g(t->device);
    sync_and_check(t);
  });
}

int ials_trainer_step(ials_trainer *t, const ials_solver_config *solver) {
  int st = ials_trainer_step_async(t, solver);
  if (st != IALS_OK) return st;
  return ials_trainer_sync(t);
}

int ials_trainer_step_io(ials_trainer *t, const ials_solver_config *solver, const float *user_in,
                         const float *item_in, float *user_out, float *item_out) {
  return guarded([&] {
    require(t != nullptr, "trainer is null");
    check_solver(solver);
    require((t->U == 0 || (user_in && user_out)) && (t->I == 0 || (item_in && item_out)),
            "factor pointer is null");
    if (t->sharded) throw std::runtime_error("sharded trainer: drive the epoch with gram_partial / solve_shard");
    if (!t->has_X) throw std::runtime_error("this trainer was restored without its interaction matrix; it cannot train");
    check_feature_solver(t, solver);
    check_feature_weight_shapes(t, false);  // before the uploads: a rejected call leaves the factors as they were
    DeviceGuard g(t->device);
    ensure_copy_stream(t);
    // item first: the user half-epoch starts with Gram(item)
    if (t->I) rows_to_device(t->factor[1].get(), t->ld, item_in, t->K, t->I, t->stream);
    // the user factors are only the warm starts of the user rows: with the CG kernels of the
    // 128-column layout they arrive while the half-epoch runs (enqueue_flagged_user_upload)
    const bool overlap_upload = solver->solver_type == IALS_SOLVER_CG && t->ld == 128 && t->U > 0 &&
                                !side_uses_features(t, 0);
    if (overlap_upload) {
      enqueue_flagged_user_upload(t, 0, t->U, user_in);
    } else if (t->U) {
      rows_to_device(t->factor[0].get(), t->ld, user_in, t->K, t->U, t->stream);
    }
    prof_mark(t);
    for (int side = 0; side < 2; side++) {  // IALSTrainer.hpp:784-787
      const DeviceCsr &csr = side == 0 ? t->X : t->Xt;
      SolveArgs a = make_args(t, side, t->factor[side].get(), csr, solver);
      if (side == 0) consume_flagged_upload(t, solver, a, 0);
      epoch_side(t, side, solver, &a);
      if (side == 1) t->epoch++;
      if (side == 0 && t->U) {
        // the new user factors are final: they travel back while the item half-epoch runs
        CUDA_CHECK(cudaEventRecord(t->users_done, t->stream));
        CUDA_CHECK(cudaStreamWaitEvent(t->copy_stream, t->users_done, 0));
        rows_to_host(user_out, t->K, t->factor[0].get(), t->ld, t->U, t->copy_stream);
      }
    }
    if (t->I) rows_to_host(item_out, t->K, t->factor[1].get(), t->ld, t->I, t->stream);
    CUDA_CHECK(cudaStreamSynchronize(t->copy_stream));
    sync_and_check(t);
  });
}

int ials_trainer_half_step(ials_trainer *t, int side, const ials_solver_config *solver) {
  return guarded([&] {
    require(t != nullptr, "trainer is null");
    require_side(side);
    check_solver(solver);
    DeviceGuard g(t->device);
    half_step(t, side, solver);
    sync_and_check(t);
  });
}

int ials_trainer_gram(ials_trainer *t, int side, float *out_host) {
  return guarded([&] {
    require(t != nullptr && out_host != nullptr, "null argument");
    require_side(side);
    DeviceGuard g(t->device);
    gram_side(t, side);
    rows_to_host(out_host, t->K, t->P[side].get(), t->ld, t->K, t->stream);
    CUDA_CHECK(cudaStreamSynchronize(t->stream));
  });
}

int ials_trainer_get_factors(ials_trainer *t, int side, float *out_host) {
  return guarded([&] {
    require(t != nullptr, "trainer is null");
    require_side(side);
    const int64_t n = t->n_rows(side);
    if (n == 0) return;
    require(out_host != nullptr, "out is null");
    DeviceGuard g(t->device);
    rows_to_host(out_host, t->K, t->factor[side].get(), t->ld, n, t->stream);
    CUDA_CHECK(cudaStreamSynchronize(t->stream));
  });
}

int ials_trainer_set_factors(ials_trainer *t, int side, const float *in_host) {
  return guarded([&] {
    require(t != nullptr, "trainer is null");
    require_side(side);
    const int64_t n = t->n_rows(side);
    if (n == 0) return;
    require(in_host != nullptr, "input is null");
    DeviceGuard g(t->device);
    rows_to_device(t->factor[side].get(), t->ld, in_host, t->K, n, t->stream);
    CUDA_CHECK(cudaStreamSynchronize(t->stream));
  });
}

int ials_trainer_set_factor_rows(ials_trainer *t, int side, int64_t row_begin, int64_t n_rows,
                                 const float *in_host, int push_to_peers) {
  return guarded([&] {
    require(t != nullptr, "trainer is null");
    require_side(side);
    require(row_begin >= 0 && n_rows >= 0 && row_begin + n_rows <= t->n_rows(side), "row range out of bounds");
    if (n_rows == 0) return;
    require(in_host != nullptr, "input is null");
    DeviceGuard g(t->device);
    float *dst = t->factor[side].get() + row_begin * t->ld;
    rows_to_device(dst, t->ld, in_host, t->K, n_rows, t->stream);
    if (push_to_peers)
      for (int p = 0; p < t->n_peers[side]; p++)
        CUDA_CHECK(cudaMemcpyAsync(t->peers[side][p] + row_begin * t->ld, dst, sizeof(float) * n_rows * t->ld,
                                   cudaMemcpyDefault, t->stream));
  });
}

int ials_trainer_set_user_rows_flagged(ials_trainer *t, int64_t row_begin, int64_t n_rows, const float *in_host) {
  return guarded([&] {
    require(t != nullptr, "trainer is null");
    require(t->has_X, "this trainer holds no interaction matrix");
    require(row_begin == t->X.row_base && n_rows == t->X.n_rows,
            "a flagged upload covers exactly the user rows this trainer solves");
    if (n_rows == 0) return;
    require(in_host != nullptr, "input is null");
    DeviceGuard g(t->device);
    enqueue_flagged_user_upload(t, row_begin, n_rows, in_host);
  });
}

int ials_trainer_get_factor_rows(ials_trainer *t, int side, int64_t row_begin, int64_t n_rows,
                                 float *out_host) {
  return guarded([&] {
    require(t != nullptr, "trainer is null");
    require_side(side);
    require(row_begin >= 0 && n_rows >= 0 && row_begin + n_rows <= t->n_rows(side), "row range out of bounds");
    if (n_rows == 0) return;
    require(out_host != nullptr, "out is null");
    DeviceGuard g(t->device);
    rows_to_host(out_host, t->K, t->factor[side].get() + row_begin * t->ld, t->ld, n_rows, t->stream);
    CUDA_CHECK(cudaStreamSynchronize(t->stream));
  });
}

int ials_trainer_factors_device(ials_trainer *t, int side, float **d_ptr, int64_t *n_rows,
                                int64_t *K, int64_t *ld) {
  return guarded([&] {
    require(t != nullptr, "trainer is null");
    require_side(side);
    if (d_ptr) *d_ptr = t->factor[side].get();
    if (n_rows) *n_rows = t->n_rows(side);
    if (K) *K = t->K;
    if (ld) *ld = t->ld;
  });
}

int ials_trainer_transform(ials_trainer *t, int side, int64_t n_rows, int64_t n_cols,
                           const int64_t *indptr, const int32_t *indices, const float *data,
                           const ials_solver_config *solver, float *out_host) {
  return guarded([&] {
    require(t != nullptr, "trainer is null");
    require_side(side);
    check_solver(solver);
    require(n_rows >= 0 && n_cols >= 0, "negative shape");
    // Solver::X_to_vector shape check, IALSTrainer.hpp:126-131
    if (side == 0 && n_cols != t->I)
      throw InvalidArgument("Shape mismatch: X.cols() = " + std::to_string(n_cols) +
                            " but other.factor.rows() = " + std::to_string(t->I) + ".");
    if (side == 1 && n_rows != t->U)
      throw InvalidArgument("Shape mismatch: X.cols() = " + std::to_string(n_rows) +
                            " but other.factor.rows() = " + std::to_string(t->U) + ".");
    DeviceGuard g(t->device);
    fold_in(t, side, n_rows, n_cols, indptr, indices, data, solver, out_host);
  });
}

int ials_trainer_compute_loss(ials_trainer *t, const ials_solver_config *solver, float *out) {
  return guarded([&] {
    require(t != nullptr && out != nullptr, "null argument");
    require(solver != nullptr && solver->n_threads > 0, "n_threads must be strictly positive.");
    if (!t->has_X) throw std::runtime_error("this trainer was restored without its interaction matrix");
    if (t->sharded) throw NotImplemented("compute_loss on a row-sharded trainer is not implemented");
    check_feature_weight_shapes(t, true);
    DeviceGuard g(t->device);
    gram_side(t, 0);
    gram_side(t, 1);
    const float bias = t->cfg.loss_type == IALS_LOSS_IALSPP ? 0.f : t->cfg.alpha0;
    // feature-aware sides are regularised towards their stored prior (:919-939); unlike step this
    // does not look at the warm-up epochs
    const float *prior[2] = {nullptr, nullptr};
    for (int side = 0; side < 2; side++)
      if (t->feature_aware && t->feat[side].n_w > 0) prior[side] = stored_prior(t, side);
    launch_loss(t->factor[0].get(), t->factor[1].get(), t->U, t->I, t->K, t->ld, t->X, t->Xt, t->P[0].get(),
                t->P[1].get(), t->cfg.alpha0, t->cfg.reg, t->cfg.nu, bias, prior[0], prior[1], t->d_loss.get(),
                t->stream);
    for (int side = 0; side < 2; side++)
      if (prior[side])
        launch_loss_add_sumsq(t->feat[side].weight.get(), t->feat[side].n_w * t->ld, t->feat[side].lambda,
                              t->d_loss.get(), t->stream);
    launch_loss_halve(t->d_loss.get(), t->stream);
    double h = 0;
    CUDA_CHECK(cudaMemcpyAsync(&h, t->d_loss.get(), sizeof(double), cudaMemcpyDeviceToHost, t->stream));
    CUDA_CHECK(cudaStreamSynchronize(t->stream));
    *out = (float)h;
  });
}

}  // extern "C"
