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
    DeviceGuard g(t->device);
    const DeviceCsr &csr = side == 0 ? t->X : t->Xt;
    SolveArgs a = make_args(t, side, t->factor[side].get(), csr, solver);
    a.n_peers = t->n_peers[side];
    for (int p = 0; p < a.n_peers; p++) a.peers[p] = t->peers[side][p];
    if (side == 0) consume_flagged_upload(t, solver, a, csr.row_base);
    run_solver(t, a, csr, solver, t->stream);
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
