// Per-row solvers of a half-epoch behind the C ABI: the solver dispatch, the tensor-core Cholesky
// and iALS++ routes over every row's Gram jobs, and the flagged upload of warm starts (step_io).
#include <algorithm>
#include <cstdlib>
#include <string>
#include <vector>

#include "trainer.cuh"

using namespace ials;

namespace ials {  // cholesky_ll.cu: Cholesky rows whose Gram blocks are in a workspace
size_t cholesky_ll_scratch_bytes();
void launch_solve_cholesky_from_gram(const SolveArgs &a, const int32_t *first_job, int job0, int job_cap,
                                     const float *workspace, float *scratch, cudaStream_t s);
}  // namespace ials

namespace {

// Solver::step_cholesky for 256-column factors with the rank updates (IALSTrainer.hpp:37-58,
// 301-308) on the tensor cores.  Per chunk of <= JC jobs one launch of wgram256_kernel
// fills  W [JC][256][256] | b [JC][8][256]  (G = W + W^T) and the left-looking Cholesky
// (cholesky_ll.cu) starts its block rows from P + G.  Rows without
// interactions are left to the plain kernel (their solution is zero).  Returns false when the
// route does not apply (negative stored values: the sqrt-weighted Gram does not exist).
// jobs per chunk: the factorisation kernel runs 592 rows at a time, so a chunk of 4096 rows ends in a
// seventh, half-empty wave (7 % of its time); 16384 jobs = 4.4 GB of workspace, fewer for smaller sides
constexpr int64_t kCholJobCapMax = 16384;
// Every row with interactions as a list of Gram jobs (<= IALS_HEAVY_JOB_LEN entries each), in the
// degree-sorted order of `csr` (the trainer's X or Xt): the schedule of the routes that form the
// normal equations on the tensor cores.
const JobPlan &all_rows_plan(ials_trainer *t, const DeviceCsr &csr, int side, cudaStream_t s) {
  JobPlan &plan = t->all_rows[side];
  std::vector<int32_t> &first = t->all_rows_first[side];
  if (first.empty()) {
    build_heavy_plan(csr, /*threshold=*/0, heavy_job_len(), plan, s);
    first.assign((size_t)plan.n_heavy + 1, 0);
    if (plan.n_heavy > 0)
      CUDA_CHECK(cudaMemcpy(first.data(), plan.heavy_first_job.get(), sizeof(int32_t) * (plan.n_heavy + 1),
                            cudaMemcpyDeviceToHost));
  }
  return plan;
}

// The rows of the all-rows plan in chunks of whole rows whose jobs fit a workspace of `cap` jobs
// (W, bpart); per chunk launch(w, h0, h1, j0): w is the weighted Gram of the jobs [j0, ...) of the
// scheduled rows [h0, h1).
template <class F>
void for_each_chunk(const ials_trainer *t, const DeviceCsr &csr, int side, const SolveArgs &a, int64_t cap,
                    float *W, float *bpart, const char *too_big, F &&launch) {
  const JobPlan &plan = t->all_rows[side];
  const std::vector<int32_t> &first = t->all_rows_first[side];
  for (int64_t h0 = 0; h0 < plan.n_heavy;) {
    int64_t h1 = h0 + 1;  // at least one row (a row has at most max_degree / job_len + 1 jobs)
    while (h1 < plan.n_heavy && first[h1 + 1] - first[h0] <= cap) h1++;
    const int j0 = first[h0], nj = first[h1] - first[h0];
    if (nj > cap) throw NotImplemented(too_big);
    WGramArgs w{};
    w.Y = a.other;
    w.ld = a.ld;
    w.indices = csr.indices.get();
    w.weights = csr.data.get();
    w.job_begin = plan.job_begin.get() + j0;
    w.job_end = plan.job_end.get() + j0;
    w.n_jobs = nj;
    w.bias = a.bias;
    w.W = W;
    w.bpart = bpart;
    launch(w, h0, h1, j0);
    h0 = h1;
  }
}

bool solve_cholesky_tensor(ials_trainer *t, const SolveArgs &a, const DeviceCsr &csr, int side,
                           cudaStream_t s) {
  if (csr.has_negative) return false;
  const JobPlan &plan = all_rows_plan(t, csr, side, s);
  const int64_t per_job = 256 * 256 + kWGram256BParts * 256;
  float *ws = t->chol_ws.ensure(std::min<int64_t>(kCholJobCapMax, std::max<int64_t>(plan.n_jobs, 1)) * per_job);
  const int kCholJobCap = (int)(t->chol_ws.size() / per_job);
  if (t->chol_scratch.get() == nullptr) {
    t->chol_scratch.alloc(cholesky_ll_scratch_bytes());
    CUDA_CHECK(cudaMemsetAsync(t->chol_scratch.get(), 0, cholesky_ll_scratch_bytes(), s));  // the padding words stay finite
  }
  float *scratch = reinterpret_cast<float *>(t->chol_scratch.get());
  for_each_chunk(t, csr, side, a, kCholJobCap, ws, ws + (size_t)kCholJobCap * 256 * 256,
                 "Cholesky on tensor cores: a row with more jobs than the workspace holds",
                 [&](const WGramArgs &w, int64_t h0, int64_t h1, int j0) {
                   launch_wgram256(w, s);
                   SolveArgs g = a;
                   g.order = csr.order.get() + h0;
                   g.n_sched = h1 - h0;
                   launch_solve_cholesky_from_gram(g, plan.heavy_first_job.get() + h0, j0, kCholJobCap, ws,
                                                   scratch, s);
                 });
  if (plan.n_heavy < a.n_sched) {  // rows without interactions: A = P + reg I, b = 0
    SolveArgs rest = a;
    rest.order = csr.order.get() + plan.n_heavy;
    rest.n_sched = a.n_sched - plan.n_heavy;
    launch_solve_cholesky_tile(rest, s);
  }
  return true;
}

// Solver::step_ialspp (IALSTrainer.hpp:387-535) for 128-column factors: per chunk of <= 4096 jobs
// one wgram_kernel launch forms G = sum c y y^T and b of every row of the chunk on the tensor cores
// (one pass over the neighbours), ialspp_dense_kernel runs the block Gauss-Seidel sweeps on
// A = P + G + reg I (ialspp_dense.cu has the algebra).  Returns false when the route does not apply.
bool solve_ialspp_tensor(ials_trainer *t, const SolveArgs &a, const DeviceCsr &csr, int side, int S, int iters,
                         cudaStream_t s) {
  if (!ialspp_dense_supported(a, S)) return false;
  if (csr.has_negative) return false;
  const JobPlan &plan = all_rows_plan(t, csr, side, s);
  // jobs per chunk (64 KB of W per job): 4096 measured 46.5 ms per ML-20M epoch against 58.5 with
  // 1024 (whose W round trip stays inside the L2, but whose launches end in half-empty waves) and
  // 46.5 with 16384 (r02al / r02am)
  const int64_t cap = 4096;
  float *W = t->gs_ws.ensure((size_t)cap * (128 * 128 + kWGramBParts * 128));
  float *bpart = W + (size_t)cap * 128 * 128;
  DenseSolveArgs d{};
  d.base = a;
  d.W = W;
  d.bpart = bpart;
  for_each_chunk(t, csr, side, a, cap, W, bpart,
                 "iALS++ on tensor cores: a row with more jobs than the workspace holds",
                 [&](const WGramArgs &w, int64_t h0, int64_t h1, int j0) {
                   launch_wgram(w, s);
                   d.base.order = csr.order.get() + h0;
                   d.n_heavy = h1 - h0;
                   d.heavy_first_job = plan.heavy_first_job.get() + h0;
                   d.job0 = j0;
                   launch_ialspp_dense(d, S, iters, s);
                 });
  if (plan.n_heavy < a.n_sched) {  // rows without interactions: A = P + reg I, b = 0
    d.base.order = csr.order.get() + plan.n_heavy;
    d.n_heavy = a.n_sched - plan.n_heavy;
    d.heavy_first_job = nullptr;
    d.job0 = 0;
    launch_ialspp_dense(d, S, iters, s);
  }
  return true;
}

// Every solve except the CG route of 128-column factors: one phase, which run_solver times.
void solve_unphased(ials_trainer *t, const SolveArgs &a, const DeviceCsr &csr, const ials_solver_config *sc,
                    cudaStream_t s) {
  if (a.n_sched == 0) return;
  if (a.prior != nullptr) {
    // feature-aware rows (step_cg with a prior / step_cholesky_with_prior, :170-271, :333-385):
    // the generic kernels, which take the prior
    if (sc->solver_type == IALS_SOLVER_CG) {
      launch_solve_cg_simple(a, s);
    } else if (sc->solver_type == IALS_SOLVER_CHOLESKY) {
      if (!cholesky_tile_supported(a)) throw NotImplemented("Cholesky solver: n_components > 256 not supported");
      launch_solve_cholesky_tile(a, s);
    } else {
      throw InvalidArgument("Feature-aware iALS does not support IALSPP.");  // :660-662
    }
    return;
  }
  const bool own_matrix = &csr == &t->X || &csr == &t->Xt;
  const int side = &csr == &t->X ? 0 : 1;
  if (sc->solver_type == IALS_SOLVER_IALSPP) {  // Solver::step_ialspp, IALSTrainer.hpp:520-535
    const int64_t S = std::min<int64_t>(sc->ialspp_subspace_dimension, a.K);
    if (!ialspp_block_supported((int)S))
      throw NotImplemented("iALS++: subspace blocks of more than 256 dimensions are not supported");
    // 128-column factors, blocks of <= 64 dimensions, the trainer's own matrix: Gram on the tensor
    // cores + block Gauss-Seidel; the per-block SIMT kernels below keep the other cases (wider
    // factors or blocks, fold-in matrices, negative stored values).  r02aj A/B on a quarter of
    // ML-20M: 139.4 ms per epoch below, 24.5 ms here (now 6.5).
    if (own_matrix && solve_ialspp_tensor(t, a, csr, side, (int)S, (int)sc->ialspp_iteration, s)) return;
    float *pred = nullptr;
    CUDA_CHECK(cudaMallocAsync(&pred, sizeof(float) * std::max<int64_t>(csr.nnz, 1), s));
    try {
      for (int64_t iter = 0; iter < sc->ialspp_iteration; iter++) {
        launch_ialspp_predict(a, pred, s);
        for (int64_t d0 = 0; d0 < a.K; d0 += S)
          launch_ialspp_block(a, pred, (int)d0, (int)std::min<int64_t>(S, a.K - d0), s);
      }
    } catch (...) {
      cudaFreeAsync(pred, s);
      throw;
    }
    CUDA_CHECK(cudaFreeAsync(pred, s));
    return;
  }
  if (sc->solver_type != IALS_SOLVER_CG) {
    // 256-column factors: rank updates on the tensor cores + left-looking factorisation
    // (IALS_CHOL=simt keeps the register-tiled SIMT kernel, for A/B runs)
    static const bool tensor_chol = [] {
      const char *e = std::getenv("IALS_CHOL");
      return e == nullptr || std::string(e) != "simt";
    }();
    if (tensor_chol && a.ld == 256 && own_matrix && solve_cholesky_tensor(t, a, csr, side, s)) return;
    if (!cholesky_tile_supported(a)) throw NotImplemented("Cholesky solver: n_components > 256 not supported");
    launch_solve_cholesky_tile(a, s);
    return;
  }
  launch_solve_cg_simple(a, s);  // ranks above 128: the generic warp-per-row kernel
}

constexpr int kReadyShift = 12;  // 4096 rows = 2 MB per chunk of a flagged upload

}  // namespace

namespace ials {

SolveArgs make_args(ials_trainer *t, int side, float *target, const DeviceCsr &csr,
                    const ials_solver_config *sc) {
  SolveArgs a{};
  a.target = target;
  a.other = t->factor[1 - side].get();
  a.P = t->P[side].get();
  a.indptr = csr.indptr.get();
  a.indices = csr.indices.get();
  a.data = csr.data.get();
  a.order = csr.order.get();
  a.n_rows = csr.n_rows;
  a.n_sched = csr.n_rows;
  a.row_base = csr.row_base;
  a.n_other = t->n_rows(1 - side);
  a.K = t->K;
  a.ld = t->ld;
  a.alpha0 = t->cfg.alpha0;
  a.reg = t->cfg.reg;
  a.nu = t->cfg.nu;
  a.bias = t->cfg.loss_type == IALS_LOSS_IALSPP ? 0.f : t->cfg.alpha0;  // IALSTrainer.hpp:190-191
  a.max_cg_steps = sc->max_cg_steps == 0 ? t->K : (int)sc->max_cg_steps;  // :232-234
  a.err_flags = t->err_flags.get();
  a.work_counter = t->work_counter.get();
  a.n_peers = 0;
  return a;
}

// Records three phase marks per call: the CG route of 128-column factors times its heavy rows
// (Gram, dense CG) and its light rows apart; every other solve is one phase after two empty ones.
void run_solver(ials_trainer *t, const SolveArgs &a, const DeviceCsr &csr,
                const ials_solver_config *sc, cudaStream_t s) {
  if (a.n_sched == 0 || a.prior != nullptr || sc->solver_type != IALS_SOLVER_CG || a.ld != 128) {
    prof_mark(t);
    prof_mark(t);
    solve_unphased(t, a, csr, sc, s);
    prof_mark(t);
    return;
  }
  const int64_t n_heavy = (csr.heavy.n_heavy > 0 && !csr.has_negative) ? csr.heavy.n_heavy : 0;
  auto run_heavy = [&] {
    if (n_heavy == 0) {
      prof_mark(t);
      prof_mark(t);
      return;
    }
    // heavy rows: tensor-core Gram of the gathered neighbours + dense CG
    const JobPlan &plan = csr.heavy;
    t->heavy_W.ensure((size_t)plan.n_jobs * 128 * 128);
    t->heavy_b.ensure((size_t)plan.n_jobs * kWGramBParts * 128);
    WGramArgs w{};
    w.Y = a.other;
    w.ld = a.ld;
    w.indices = csr.indices.get();
    w.weights = csr.data.get();
    w.job_begin = plan.job_begin.get();
    w.job_end = plan.job_end.get();
    w.n_jobs = plan.n_jobs;
    w.bias = a.bias;
    w.W = t->heavy_W.get();
    w.bpart = t->heavy_b.get();
    DenseSolveArgs d{};
    d.base = a;
    d.n_heavy = plan.n_heavy;
    d.heavy_first_job = plan.heavy_first_job.get();
    d.W = t->heavy_W.get();
    d.bpart = t->heavy_b.get();
    launch_wgram(w, s);
    prof_mark(t);
    launch_dense_cg(d, s);
    prof_mark(t);
  };
  auto run_light = [&] {
    SolveArgs light = a;  // everything else (all rows when a stored value is negative)
    light.order = csr.order.get() + n_heavy;
    light.n_sched = csr.n_rows - n_heavy;
    // rows whose warm starts are still arriving (step_io) are taken in arrival order
    if (a.ready_flags != nullptr && t->order_io.get() != nullptr && &csr == &t->X) light.order = t->order_io.get();
    launch_solve_cg_rows(light, s);
    prof_mark(t);
  };
  if (a.ready_flags != nullptr) {
    // the few heavy rows sit in arbitrary chunks of the upload: after the light rows every chunk
    // is there (the phase marks keep their count, not their labels, in this order)
    run_light();
    run_heavy();
  } else {
    run_heavy();
    run_light();
  }
}

void ensure_copy_stream(ials_trainer *t) {
  if (t->copy_stream == nullptr) {
    CUDA_CHECK(cudaStreamCreateWithFlags(&t->copy_stream, cudaStreamNonBlocking));
    CUDA_CHECK(cudaEventCreateWithFlags(&t->users_done, cudaEventDisableTiming));
    CUDA_CHECK(cudaEventCreateWithFlags(&t->upload_done, cudaEventDisableTiming));
  }
}

// The user rows [row_begin, row_begin + n_rows) (the whole matrix, or this rank's shard) arrive from
// the host in chunks on the copy stream WHILE the user half-epoch runs: a 4-byte copy behind every
// chunk raises its flag (the copy engine does; a flag KERNEL found no SM to run on -- cg_rows_kernel
// holds every register of every SM while its warps wait for exactly that flag: r02t, 1.7 s per
// step), a row waits for its chunk before it reads its warm start (and therefore also before it
// writes its solution, which a late chunk would overwrite), and the light rows are taken in
// (arrival chunk, descending degree) order -- in the degree-sorted order every warp blocked on a
// row of a late chunk (r02u).  Only the CG kernels of the 128-column layout wait for flags; any
// other solve first waits for upload_done.
void enqueue_flagged_user_upload(ials_trainer *t, int64_t row_begin, int64_t n_rows, const float *rows_host) {
  ensure_copy_stream(t);
  const int n_chunks = (int)((n_rows + (1ll << kReadyShift) - 1) >> kReadyShift);
  if ((size_t)n_chunks > t->ready_flags.size()) {
    t->ready_flags.alloc(n_chunks);
    t->ready_host.alloc(n_chunks);
    CUDA_CHECK(cudaMemsetAsync(t->ready_flags.get(), 0, sizeof(int) * n_chunks, t->stream));
    t->ready_token = 0;
  }
  if (t->order_io.get() == nullptr) {  // once: the light rows by (chunk of the upload, descending degree)
    const DeviceCsr &X = t->X;
    const int64_t nh = (X.heavy.n_heavy > 0 && !X.has_negative) ? X.heavy.n_heavy : 0, nl = X.n_rows - nh;
    std::vector<int32_t> ord((size_t)std::max<int64_t>(nl, 1));
    if (nl)
      CUDA_CHECK(cudaMemcpyAsync(ord.data(), X.order.get() + nh, sizeof(int32_t) * nl, cudaMemcpyDeviceToHost,
                                 t->stream));
    CUDA_CHECK(cudaStreamSynchronize(t->stream));
    ord.resize((size_t)nl);
    // X.order is by descending degree: a stable sort by chunk keeps that order inside a chunk
    // (CSR row u is factor row X.row_base + u, and the upload starts at X.row_base)
    std::stable_sort(ord.begin(), ord.end(),
                     [&](int32_t x, int32_t y) { return (x >> kReadyShift) < (y >> kReadyShift); });
    t->order_io.alloc(std::max<int64_t>(nl, 1));
    if (nl) CUDA_CHECK(cudaMemcpy(t->order_io.get(), ord.data(), sizeof(int32_t) * nl, cudaMemcpyHostToDevice));
  }
  t->ready_token++;  // never 0; a stale flag of an earlier step never matches
  // the flags' reset (first use) and every kernel enqueued so far precede the copies
  CUDA_CHECK(cudaEventRecord(t->users_done, t->stream));
  CUDA_CHECK(cudaStreamWaitEvent(t->copy_stream, t->users_done, 0));
  for (int c = 0; c < n_chunks; c++) {
    const int64_t r0 = (int64_t)c << kReadyShift, nr = std::min<int64_t>(1ll << kReadyShift, n_rows - r0);
    rows_to_device(t->factor[0].get() + (row_begin + r0) * t->ld, t->ld, rows_host + r0 * t->K, t->K, nr,
                   t->copy_stream);
    t->ready_host.get()[c] = t->ready_token;
    CUDA_CHECK(cudaMemcpyAsync(t->ready_flags.get() + c, t->ready_host.get() + c, sizeof(int),
                               cudaMemcpyHostToDevice, t->copy_stream));
  }
  CUDA_CHECK(cudaEventRecord(t->upload_done, t->copy_stream));
  t->ready_pending = true;
}

// Give the pending flagged upload to the user solve `a` (if its kernels can wait for flags), or make
// the stream wait for the whole upload.
void consume_flagged_upload(ials_trainer *t, const ials_solver_config *sc, SolveArgs &a, int64_t row_begin) {
  if (!t->ready_pending) return;
  t->ready_pending = false;
  if (sc->solver_type == IALS_SOLVER_CG && t->ld == 128 && a.prior == nullptr) {
    a.ready_flags = t->ready_flags.get();
    a.ready_token = t->ready_token;
    a.ready_shift = kReadyShift;
    a.ready_base = row_begin;
  } else {
    CUDA_CHECK(cudaStreamWaitEvent(t->stream, t->upload_done, 0));
  }
}

}  // namespace ials
