// Feature-aware iALS behind the C ABI (IALSTrainer.hpp:634-662, 758-789, 1001-1209): feature
// upload, the stored prior, the ridge refit of the feature weights and their entry points.
#include <cmath>
#include <string>
#include <vector>

#include "trainer.cuh"

using namespace ials;

namespace {

// host features -> device (dense row-major when indptr == nullptr, else CSR) into a fresh `owner`,
// which keeps the arrays
void upload_features(ials_trainer::FeatureSide &owner, int64_t n_rows, int64_t n_cols, const float *dense,
                     const int64_t *indptr, const int32_t *indices, const float *data) {
  FeatureDev &F = owner.F;
  F.n_rows = n_rows;
  F.n_cols = n_cols;
  if (indptr == nullptr) {
    require(dense != nullptr || n_rows * n_cols == 0, "feature matrix is null");
    F.dense = owner.dense.alloc(std::max<int64_t>(n_rows * n_cols, 1));
    if (n_rows * n_cols)
      CUDA_CHECK(cudaMemcpy(owner.dense.get(), dense, sizeof(float) * n_rows * n_cols, cudaMemcpyHostToDevice));
    return;
  }
  require(indptr[0] == 0, "feature indptr must start at 0");
  const int64_t nnz = indptr[n_rows];
  require(nnz == 0 || (indices != nullptr && data != nullptr), "feature indices / data are null");
  for (int64_t j = 0; j < nnz; j++) require(indices[j] >= 0 && indices[j] < n_cols, "feature column out of range");
  copy_csr(owner.csr, n_rows, n_cols, nnz, indptr, indices, data, cudaMemcpyHostToDevice);
  F.nnz = nnz;
  F.indptr = owner.csr.indptr.get();
  F.indices = owner.csr.indices.get();
  F.data = owner.csr.data.get();
}

// initialize_feature_aware (:1001-1014) for the rows the trainer holds of the side's interaction
// matrix (all of them, or a rank's shard); records whether one of those rows is empty
void init_features(ials_trainer *t, int side, int64_t n_rows, int64_t n_cols, const float *dense,
                   const int64_t *indptr, const int32_t *indices, const float *data, float lambda_feature,
                   int64_t feature_warmup_epochs) {
  if (!t->has_X) throw std::runtime_error("this trainer was restored without its interaction matrix");
  const DeviceCsr &csr = side == 0 ? t->X : t->Xt;
  if (n_rows != csr.n_rows) throw InvalidArgument("Feature matrix row count mismatch.");
  if (n_cols > 0 && !(lambda_feature > 0.f))
    throw InvalidArgument("Feature weight regularization must be positive.");
  DeviceGuard g(t->device);
  ials_trainer::FeatureSide &f = t->feat[side];
  f = ials_trainer::FeatureSide{};
  upload_features(f, n_rows, n_cols, dense, indptr, indices, data);
  f.given = f.weight_set = true;
  f.n_w = n_cols;
  f.lambda = lambda_feature;
  CUDA_CHECK(cudaMemset(f.weight.alloc(std::max<int64_t>(n_cols * t->ld, 1)), 0,
                        sizeof(float) * std::max<int64_t>(n_cols * t->ld, 1)));  // setZero, :1012
  {  // does the side's interaction matrix have an empty row? (step_with_prior's guard)
    std::vector<int64_t> ip((size_t)csr.n_rows + 1);
    CUDA_CHECK(cudaMemcpy(ip.data(), csr.indptr.get(), sizeof(int64_t) * (csr.n_rows + 1), cudaMemcpyDeviceToHost));
    f.has_empty_row = false;
    for (int64_t r = 0; r < csr.n_rows; r++)
      if (ip[r] == ip[r + 1]) {
        f.has_empty_row = true;
        break;
      }
  }
  t->feature_aware = true;
  t->feature_warmup = feature_warmup_epochs;
}

const char *side_name(int side) { return side == 0 ? "user" : "item"; }
const char *side_Name(int side) { return side == 0 ? "User" : "Item"; }

// validate_user_feature_matrix / validate_item_feature_matrix (:1016-1042)
void validate_feature_cols(const ials_trainer *t, int side, int64_t cols) {
  const ials_trainer::FeatureSide &f = t->feat[side];
  if (!f.weight_set) throw InvalidArgument(std::string(side_Name(side)) + " feature weights are not initialized.");
  if (cols != f.n_w)
    throw InvalidArgument(std::string("Shape mismatch: ") + side_name(side) + " feature matrix has " +
                          std::to_string(cols) + " columns but " + side_name(side) + "_feature_weight has " +
                          std::to_string(f.n_w) + " rows.");
}

}  // namespace

namespace ials {

// step_with_prior's guard (:639-652): with alpha0 = 0 and a vanishing ridge an empty row has no
// unique solution
void check_prior_defined(const ials_trainer *t, int side, bool has_empty_row) {
  if (t->cfg.alpha0 != 0.f) return;
  const float r0 = t->cfg.reg * std::pow(t->cfg.alpha0 * (float)t->n_rows(1 - side) + 0.f, t->cfg.nu);
  if ((!(r0 > 0.f) || !std::isfinite(r0)) && has_empty_row)
    throw InvalidArgument("Feature-prior embedding is not uniquely defined for an empty interaction row when "
                          "alpha0 and its regularization are zero.");
}

bool side_uses_features(const ials_trainer *t, int side) {
  return t->feature_aware && t->epoch >= t->feature_warmup && t->feat[side].n_w > 0;
}

// The stored features meet the stored weight in the prior F W and in the weight refit, which read
// F.n_cols rows of the weight and of its cached Gram factor.  The setter accepts any row count (as
// the reference's def_rw does), so the shape is checked where the two meet, before the first launch:
// on the sides a step uses (`any_epoch` false) or on every side with a weight (compute_loss, which
// does not look at the warm-up).
void check_feature_weight_shapes(const ials_trainer *t, bool any_epoch) {
  for (int side = 0; side < 2; side++) {
    const bool used = any_epoch ? t->feature_aware && t->feat[side].n_w > 0 : side_uses_features(t, side);
    if (used) validate_feature_cols(t, side, t->feat[side].F.n_cols);
  }
}

// stored_user_feature_prior / stored_item_feature_prior (:1044-1050) into feat[side].prior: one row
// per feature row (every row of the side, or a rank's own rows)
const float *stored_prior(ials_trainer *t, int side) {
  ials_trainer::FeatureSide &f = t->feat[side];
  const int64_t n = f.F.n_rows;
  launch_feature_prior(f.F, f.weight.get(), t->ld, f.prior.ensure(std::max<int64_t>(n * t->ld, 1)), t->stream);
  return f.prior.get();
}

// update_stored_*_feature_weight -> update_feature_weight (:1052-1064, 1182-1209)
void update_feature_weight(ials_trainer *t, int side) {
  ials_trainer::FeatureSide &f = t->feat[side];
  if (f.n_w == 0) return;
  const DeviceCsr &csr = side == 0 ? t->X : t->Xt;
  const int64_t n = t->n_rows(side);
  if (!f.cache_ready) {  // initialize_feature_weight_cache (:1083-1132): once per trainer
    f.rw.ensure(std::max<int64_t>(n, 1));
    f.llt.ensure(f.n_w * f.n_w);
    f.rhs.ensure(f.n_w * t->ld);
    launch_feature_row_weights(csr.indptr.get(), n, t->n_rows(1 - side), t->cfg.alpha0, t->cfg.reg, t->cfg.nu,
                               f.rw.get(), t->stream);
    launch_feature_gram_llt(f.F, f.rw.get(), f.lambda, f.llt.get(), t->err_flags.get() + kErrFeatureLlt, t->stream);
    f.cache_ready = true;
  }
  // solve_feature_weight (:1134-1180); the solution replaces the weight
  launch_feature_ridge_solve(f.F, f.rw.get(), t->factor[side].get(), t->ld, f.llt.get(), f.rhs.get(),
                             t->err_flags.get() + kErrFeatureSolve, t->stream);
  CUDA_CHECK(cudaMemcpyAsync(f.weight.get(), f.rhs.get(), sizeof(float) * f.n_w * t->ld, cudaMemcpyDeviceToDevice,
                             t->stream));
}

void check_feature_solver(const ials_trainer *t, const ials_solver_config *sc) {
  if (t->feature_aware && sc->solver_type == IALS_SOLVER_IALSPP)
    throw InvalidArgument("Feature-aware iALS does not support IALSPP.");  // :759-761
}

}  // namespace ials

extern "C" {

// ---- feature-aware iALS: the C ABI (wrapper.cpp:133-136, 144-155, 160-161) ----

int ials_trainer_set_features(ials_trainer *t, int side, int64_t n_rows, int64_t n_cols, const float *dense,
                              const int64_t *indptr, const int32_t *indices, const float *data,
                              float lambda_feature, int64_t feature_warmup_epochs) {
  return guarded([&] {
    require(t != nullptr, "trainer is null");
    require_side(side);
    require(n_rows >= 0 && n_cols >= 0 && feature_warmup_epochs >= 0, "negative shape");
    if (t->sharded) throw NotImplemented("feature-aware iALS on a row-sharded trainer is not implemented");
    init_features(t, side, n_rows, n_cols, dense, indptr, indices, data, lambda_feature, feature_warmup_epochs);
  });
}

int ials_trainer_set_shard_features(ials_trainer *t, int side, int64_t n_rows, int64_t n_cols, const float *dense,
                                    const int64_t *indptr, const int32_t *indices, const float *data,
                                    float lambda_feature, int64_t feature_warmup_epochs, int *has_empty_row) {
  return guarded([&] {
    require(t != nullptr, "trainer is null");
    require_side(side);
    require(n_rows >= 0 && n_cols >= 0 && feature_warmup_epochs >= 0, "negative shape");
    require(t->sharded, "not a row-sharded trainer: use ials_trainer_set_features");
    init_features(t, side, n_rows, n_cols, dense, indptr, indices, data, lambda_feature, feature_warmup_epochs);
    if (has_empty_row) *has_empty_row = t->feat[side].has_empty_row ? 1 : 0;
  });
}

int ials_trainer_feature_weight_rows(ials_trainer *t, int side, int64_t *n_rows) {
  return guarded([&] {
    require(t != nullptr && n_rows != nullptr, "null argument");
    require_side(side);
    *n_rows = t->feat[side].weight_set ? t->feat[side].n_w : 0;
  });
}

int ials_trainer_get_feature_weight(ials_trainer *t, int side, float *out_host) {
  return guarded([&] {
    require(t != nullptr, "trainer is null");
    require_side(side);
    const ials_trainer::FeatureSide &f = t->feat[side];
    if (!f.weight_set || f.n_w == 0) return;
    require(out_host != nullptr, "out is null");
    DeviceGuard g(t->device);
    CUDA_CHECK(cudaStreamSynchronize(t->stream));
    rows_to_host(out_host, t->K, f.weight.get(), t->ld, f.n_w);
  });
}

int ials_trainer_set_feature_weight(ials_trainer *t, int side, int64_t n_rows, const float *in_host) {
  return guarded([&] {
    require(t != nullptr, "trainer is null");
    require_side(side);
    require(n_rows >= 0 && (n_rows == 0 || in_host != nullptr), "null argument");
    DeviceGuard g(t->device);
    ials_trainer::FeatureSide &f = t->feat[side];
    CUDA_CHECK(cudaStreamSynchronize(t->stream));
    if (n_rows != f.n_w || f.weight.get() == nullptr) {  // def_rw assigns the whole matrix (wrapper.cpp:160-161)
      CUDA_CHECK(f.rhs.reset());
      CUDA_CHECK(f.llt.reset());
      f.cache_ready = false;
      f.weight.alloc(std::max<int64_t>(n_rows * t->ld, 1));
      f.n_w = n_rows;
    }
    CUDA_CHECK(cudaMemset(f.weight.get(), 0, sizeof(float) * std::max<int64_t>(n_rows * t->ld, 1)));
    if (n_rows) rows_to_device(f.weight.get(), t->ld, in_host, t->K, n_rows);
    f.weight_set = true;
  });
}

// transform_user_feature / transform_item_feature (:820-830): features x stored weight
int ials_trainer_transform_feature(ials_trainer *t, int side, int64_t n_rows, int64_t n_cols, const float *dense,
                                   const int64_t *indptr, const int32_t *indices, const float *data,
                                   float *out_host) {
  return guarded([&] {
    require(t != nullptr, "trainer is null");
    require_side(side);
    require(n_rows >= 0 && n_cols >= 0, "negative shape");
    validate_feature_cols(t, side, n_cols);
    if (n_rows == 0) return;
    require(out_host != nullptr, "out is null");
    DeviceGuard g(t->device);
    ials_trainer::FeatureSide tmp;
    DeviceBuffer<float> prior;
    StreamSyncOnExit sync{t->stream};
    upload_features(tmp, n_rows, n_cols, dense, indptr, indices, data);
    launch_feature_prior(tmp.F, t->feat[side].weight.get(), t->ld, prior.alloc(n_rows * t->ld), t->stream);
    rows_to_host(out_host, t->K, prior.get(), t->ld, n_rows, t->stream);
    CUDA_CHECK(cudaStreamSynchronize(t->stream));
  });
}

// transform_user_with_feature / transform_item_with_feature (:803-818): fold-in whose rows start from,
// and are regularised towards, features x stored weight (X_to_vector_with_prior, :142-167)
int ials_trainer_transform_with_feature(ials_trainer *t, int side, int64_t n_rows, int64_t n_cols,
                                        const int64_t *indptr, const int32_t *indices, const float *data,
                                        int64_t f_rows, int64_t f_cols, const float *f_dense,
                                        const int64_t *f_indptr, const int32_t *f_indices, const float *f_data,
                                        const ials_solver_config *solver, float *out_host) {
  return guarded([&] {
    require(t != nullptr, "trainer is null");
    require_side(side);
    check_solver(solver);
    require(n_rows >= 0 && n_cols >= 0 && f_rows >= 0 && f_cols >= 0, "negative shape");
    validate_feature_cols(t, side, f_cols);
    if (side == 0 && n_cols != t->I)
      throw InvalidArgument("Shape mismatch: X.cols() = " + std::to_string(n_cols) +
                            " but other.factor.rows() = " + std::to_string(t->I) + ".");
    if (side == 1 && n_rows != t->U)
      throw InvalidArgument("Shape mismatch: X.cols() = " + std::to_string(n_rows) +
                            " but other.factor.rows() = " + std::to_string(t->U) + ".");
    const int64_t n_new = side == 0 ? n_rows : n_cols;
    if (f_rows != n_new) throw InvalidArgument("Feature prior shape does not match X.");  // :153-155
    if (solver->solver_type == IALS_SOLVER_IALSPP)
      throw InvalidArgument("Feature-aware iALS does not support IALSPP.");
    DeviceGuard g(t->device);
    ials_trainer::FeatureSide tmp;  // fold_in synchronises the stream before these are freed
    DeviceBuffer<float> prior;
    fold_in(t, side, n_rows, n_cols, indptr, indices, data, solver, out_host, [&](const DeviceCsr &csr) {
      // the guard of step_with_prior needs to know whether a new row is empty
      std::vector<int64_t> ip((size_t)n_new + 1);
      CUDA_CHECK(cudaMemcpyAsync(ip.data(), csr.indptr.get(), sizeof(int64_t) * (n_new + 1), cudaMemcpyDeviceToHost,
                                 t->stream));
      CUDA_CHECK(cudaStreamSynchronize(t->stream));
      bool empty = false;
      for (int64_t r = 0; r < n_new && !empty; r++) empty = ip[r] == ip[r + 1];
      check_prior_defined(t, side, empty);
      upload_features(tmp, f_rows, f_cols, f_dense, f_indptr, f_indices, f_data);
      const size_t bytes = sizeof(float) * std::max<int64_t>(n_new * t->ld, 1);
      CUDA_CHECK(cudaMemsetAsync(prior.alloc(std::max<int64_t>(n_new * t->ld, 1)), 0, bytes, t->stream));
      launch_feature_prior(tmp.F, t->feat[side].weight.get(), t->ld, prior.get(), t->stream);
      return prior.get();
    });
  });
}

}  // extern "C"
