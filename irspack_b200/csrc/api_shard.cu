// Row-sharded multi-GPU trainer behind the C ABI: a rank solves its own rows of X / X^T against
// full factor replicas, shares its Gram partial and exchanges factor rows through CUDA IPC.
#include <cstring>

#include "trainer.cuh"

using namespace ials;

extern "C" {

int ials_trainer_create_sharded(const ials_model_config *config, int64_t n_users, int64_t n_items,
                                int64_t user_begin, int64_t user_end, const int64_t *u_indptr,
                                const int32_t *u_indices, const float *u_data, int64_t item_begin,
                                int64_t item_end, const int64_t *i_indptr, const int32_t *i_indices,
                                const float *i_data, int csr_on_device, int init_on_device,
                                int device, ials_trainer **out) {
  return guarded([&] {
    require(out != nullptr, "out is null");
    *out = nullptr;
    require(0 <= user_begin && user_begin <= user_end && user_end <= n_users, "bad user shard");
    require(0 <= item_begin && item_begin <= item_end && item_end <= n_items, "bad item shard");
    TrainerPtr t = new_trainer(config, n_users, n_items, device);
    DeviceGuard g(device);
    alloc_common(t.get());
    // rows [user_begin, user_end) of X and rows [item_begin, item_end) of X^T
    upload_csr(t->X, user_end - user_begin, n_items, u_indptr, u_indices, u_data, csr_on_device != 0);
    upload_csr(t->Xt, item_end - item_begin, n_users, i_indptr, i_indices, i_data, csr_on_device != 0);
    t->X.row_base = user_begin;
    t->Xt.row_base = item_begin;
    plan_csr(t.get(), t->X);
    plan_csr(t.get(), t->Xt);
    t->has_X = true;
    t->sharded = true;
    t->shard[0][0] = user_begin; t->shard[0][1] = user_end;
    t->shard[1][0] = item_begin; t->shard[1][1] = item_end;
    init_factors(t.get(), init_on_device != 0);
    *out = t.release();
  });
}

int ials_trainer_gram_partial(ials_trainer *t, int factor_side, float **d_out, int64_t *count) {
  return guarded([&] {
    require(t != nullptr, "trainer is null");
    require_side(factor_side);
    DeviceGuard g(t->device);
    const int64_t b = t->sharded ? t->shard[factor_side][0] : 0;
    const int64_t e = t->sharded ? t->shard[factor_side][1] : t->n_rows(factor_side);
    float *dst = t->P[1 - factor_side].get();
    gram_rows(t, factor_side, b, e, dst);
    if (d_out) *d_out = dst;
    if (count) *count = (int64_t)t->ld * t->ld;
  });
}

int ials_trainer_solve_shard(ials_trainer *t, int side, const ials_solver_config *solver) {
  return guarded([&] {
    require(t != nullptr, "trainer is null");
    require_side(side);
    check_solver(solver);
    if (!t->has_X) throw std::runtime_error("no interaction matrix");
    check_feature_solver(t, solver);
    check_feature_weight_shapes(t, false);
    DeviceGuard g(t->device);
    const DeviceCsr &csr = side == 0 ? t->X : t->Xt;
    SolveArgs a = make_args(t, side, t->factor[side].get(), csr, solver);
    a.n_peers = t->n_peers[side];
    for (int p = 0; p < a.n_peers; p++) a.peers[p] = t->peers[side][p];
    ials_trainer::FeatureSide &f = t->feat[side];
    f.refit_pending = side_uses_features(t, side);  // IALSTrainer.hpp:762, 777
    if (f.refit_pending) {
      check_prior_defined(t, side, f.has_empty_row);
      // the kernels read the prior of factor row gu at prior[gu * ld]; the buffer holds the shard's rows
      a.prior = stored_prior(t, side) - csr.row_base * t->ld;
    }
    if (side == 0) consume_flagged_upload(t, solver, a, csr.row_base);
    run_solver(t, a, csr, solver, t->stream);
    if (side == 1) t->epoch++;  // the item half ends the epoch (:788)
  });
}

int ials_trainer_check_shard_step(ials_trainer *t, const ials_solver_config *solver, int user_has_empty_row,
                                  int item_has_empty_row) {
  return guarded([&] {
    require(t != nullptr, "trainer is null");
    check_solver(solver);
    check_feature_solver(t, solver);
    check_feature_weight_shapes(t, false);
    const bool empty[2] = {user_has_empty_row != 0, item_has_empty_row != 0};
    for (int side = 0; side < 2; side++)
      if (side_uses_features(t, side)) check_prior_defined(t, side, empty[side]);
  });
}

int ials_trainer_feature_partials(ials_trainer *t, int side, float **d_gram, int64_t *gram_count, float **d_rhs,
                                  int64_t *rhs_count) {
  return guarded([&] {
    require(t != nullptr && d_gram != nullptr && gram_count != nullptr && d_rhs != nullptr && rhs_count != nullptr,
            "null argument");
    require_side(side);
    require(t->sharded, "not a row-sharded trainer");
    *d_gram = *d_rhs = nullptr;
    *gram_count = *rhs_count = 0;
    ials_trainer::FeatureSide &f = t->feat[side];
    if (!f.refit_pending) return;
    DeviceGuard g(t->device);
    const DeviceCsr &csr = side == 0 ? t->X : t->Xt;
    if (!f.cache_ready) {  // initialize_feature_weight_cache (:1083-1132), over the shard's rows
      f.rw.ensure(std::max<int64_t>(csr.n_rows, 1));
      f.llt.ensure(f.n_w * f.n_w);
      launch_feature_row_weights(csr.indptr.get(), csr.n_rows, t->n_rows(1 - side), t->cfg.alpha0, t->cfg.reg,
                                 t->cfg.nu, f.rw.get(), t->stream);
      launch_feature_gram(f.F, f.rw.get(), f.llt.get(), t->stream);
      *d_gram = f.llt.get();
      *gram_count = f.n_w * f.n_w;
    }
    // solve_feature_weight's right-hand side (:1134-1160) over the shard's freshly solved rows
    f.rhs.ensure(f.n_w * t->ld);
    launch_feature_rhs(f.F, f.rw.get(), t->factor[side].get() + csr.row_base * t->ld, t->ld, f.rhs.get(),
                       t->stream);
    *d_rhs = f.rhs.get();
    *rhs_count = f.n_w * t->ld;
  });
}

int ials_trainer_feature_refit(ials_trainer *t, int side) {
  return guarded([&] {
    require(t != nullptr, "trainer is null");
    require_side(side);
    require(t->sharded, "not a row-sharded trainer");
    ials_trainer::FeatureSide &f = t->feat[side];
    if (!f.refit_pending) return;
    f.refit_pending = false;
    DeviceGuard g(t->device);
    if (!f.cache_ready) {
      launch_feature_llt(f.llt.get(), f.n_w, f.lambda, t->err_flags.get() + kErrFeatureLlt, t->stream);
      f.cache_ready = true;
    }
    launch_feature_solve(f.llt.get(), f.n_w, f.rhs.get(), t->ld, t->err_flags.get() + kErrFeatureSolve, t->stream);
    CUDA_CHECK(cudaMemcpyAsync(f.weight.get(), f.rhs.get(), sizeof(float) * f.n_w * t->ld, cudaMemcpyDeviceToDevice,
                               t->stream));
  });
}

int ials_trainer_compute_loss_shard(ials_trainer *t, const ials_solver_config *solver, int include_global,
                                    double *out) {
  return guarded([&] {
    require(t != nullptr && out != nullptr, "null argument");
    require(solver != nullptr && solver->n_threads > 0, "n_threads must be strictly positive.");
    require(t->sharded, "not a row-sharded trainer: use ials_trainer_compute_loss");
    check_feature_weight_shapes(t, true);
    DeviceGuard g(t->device);
    const float *P[2] = {nullptr, nullptr};
    if (include_global) {  // sum(P_user .* P_item) / alpha0 from the full replicas
      gram_side(t, 0);
      gram_side(t, 1);
      P[0] = t->P[0].get();
      P[1] = t->P[1].get();
    }
    const float bias = t->cfg.loss_type == IALS_LOSS_IALSPP ? 0.f : t->cfg.alpha0;
    const float *prior[2] = {nullptr, nullptr};
    for (int side = 0; side < 2; side++)
      if (t->feature_aware && t->feat[side].n_w > 0) prior[side] = stored_prior(t, side);
    launch_loss_shard(t->factor[0].get(), t->factor[1].get(), t->U, t->I, t->ld, t->X, t->Xt, P[0], P[1],
                      t->cfg.alpha0, t->cfg.reg, t->cfg.nu, bias, prior[0], prior[1], t->d_loss.get(), t->stream);
    for (int side = 0; side < 2; side++)
      if (include_global && prior[side])
        launch_loss_add_sumsq(t->feat[side].weight.get(), t->feat[side].n_w * t->ld, t->feat[side].lambda,
                              t->d_loss.get(), t->stream);
    launch_loss_halve(t->d_loss.get(), t->stream);
    CUDA_CHECK(cudaMemcpyAsync(out, t->d_loss.get(), sizeof(double), cudaMemcpyDeviceToHost, t->stream));
    CUDA_CHECK(cudaStreamSynchronize(t->stream));
  });
}

int ials_trainer_shard_range(ials_trainer *t, int side, int64_t *begin, int64_t *end) {
  return guarded([&] {
    require(t != nullptr && begin != nullptr && end != nullptr, "null argument");
    require_side(side);
    *begin = t->sharded ? t->shard[side][0] : 0;
    *end = t->sharded ? t->shard[side][1] : t->n_rows(side);
  });
}

int ials_trainer_ipc_handle(ials_trainer *t, int side, unsigned char handle_out[64]) {
  return guarded([&] {
    require(t != nullptr && handle_out != nullptr, "null argument");
    require_side(side);
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    DeviceGuard g(t->device);
    cudaIpcMemHandle_t h;
    CUDA_CHECK(cudaIpcGetMemHandle(&h, t->factor[side].get()));
    std::memcpy(handle_out, &h, 64);
  });
}

int ials_trainer_ipc_open_peers(ials_trainer *t, int side, const unsigned char *handles, int world,
                                int rank) {
  return guarded([&] {
    require(t != nullptr && handles != nullptr, "null argument");
    require_side(side);
    require(world >= 1 && world <= 9 && rank >= 0 && rank < world, "world must be <= 9");
    DeviceGuard g(t->device);
    for (int p = 0; p < t->n_peers[side]; p++) cudaIpcCloseMemHandle(t->peers[side][p]);
    t->n_peers[side] = 0;
    for (int r = 0; r < world; r++) {
      if (r == rank) continue;
      cudaIpcMemHandle_t h;
      std::memcpy(&h, handles + 64 * r, 64);
      void *p = nullptr;
      CUDA_CHECK(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
      t->peers[side][t->n_peers[side]++] = (float *)p;
    }
  });
}
}  // extern "C"
