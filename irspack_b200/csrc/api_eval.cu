// Evaluation passes behind the C ABI: an evaluation set (ground truth, optional mask and allow-lists,
// cutoffs and per-cutoff accumulators, uploaded once) and one call that produces the lists of a range of
// users and accumulates their metrics without the lists leaving the device.  A row-sharded trainer runs
// it on its own users; the caller all-reduces the accumulators and reduces the merged histograms.
// A cold set holds users that are not rows of the model (EvaluatorWithColdUser, evaluator.py:470-657):
// its pass folds their input rows in on the device and ranks the results the same way.
#include <algorithm>
#include <cmath>
#include <vector>

#include "trainer.cuh"

using namespace ials;

struct ials_eval_set {
  int device = 0;
  int64_t row_begin = 0, n_rows = 0, n_items = 0;
  DeviceBuffer<int64_t> gt_indptr;  // [n_rows + 1], from 0
  DeviceBuffer<int32_t> gt_indices;
  int mask_mode = 0;                // 0: the trainer's training rows, 2: the mask below
  DeviceBuffer<int64_t> m_indptr;
  DeviceBuffer<int32_t> m_indices;
  bool mask_sorted = true;
  ListJob allow;                    // allow_n_lists / a_* of the lists (rows relative to row_begin)
  DeviceBuffer<int64_t> a_indptr;
  DeviceBuffer<int32_t> a_indices;
  std::vector<uint32_t> a_words;
  int n_cut = 0;
  int64_t kmax = 0;
  int recall_with_cutoff = 0;
  DeviceBuffer<int32_t> cutoffs;           // [n_cut]
  DeviceBuffer<double> discount, cum;      // [kmax]
  DeviceBuffer<double> sums;               // [n_cut][5] hit, recall, ndcg, map, precision
  DeviceBuffer<unsigned long long> counts; // valid_user[n_cut] | total_user[n_cut]
  DeviceBuffer<unsigned long long> hist;   // [n_cut][n_items]
  DeviceBuffer<double> partial;            // metrics kernel scratch
  DeviceBuffer<unsigned char> div_ws;
  DeviceBuffer<double> div_out;            // [3]
  // cold set: the input rows in chunks of kListSlabRows rows, each planned once (plan_csr), and the
  // slab one chunk is folded into
  bool cold = false;
  std::vector<DeviceCsr> input;
  DeviceBuffer<float> slab;
};

namespace {

void zero_accumulators(ials_eval_set *e, cudaStream_t s) {
  CUDA_CHECK(cudaMemsetAsync(e->sums.get(), 0, sizeof(double) * 5 * e->n_cut, s));
  CUDA_CHECK(cudaMemsetAsync(e->counts.get(), 0, sizeof(unsigned long long) * 2 * e->n_cut, s));
  CUDA_CHECK(cudaMemsetAsync(e->hist.get(), 0, sizeof(unsigned long long) * e->n_cut * e->n_items, s));
}

// Every cutoff in [1, n_items] and <= 1024 (evaluator.cpp:265-266); returns the largest
int64_t check_cutoffs(const ials_trainer *t, const int64_t *cutoffs, int64_t n_cutoffs) {
  require(n_cutoffs >= 1 && cutoffs != nullptr, "at least one cutoff");
  int64_t kmax = 0;
  for (int64_t c = 0; c < n_cutoffs; c++) {
    require(cutoffs[c] >= 1 && cutoffs[c] <= t->I, "cutoff must be in [1, n_items]");  // evaluator.cpp:265-266
    require(cutoffs[c] <= 1024, "k > 1024 is not supported");
    kmax = std::max(kmax, cutoffs[c]);
  }
  return kmax;
}

// The set's ground truth (n_rows rows, sorted), on stream s
void stage_ground_truth(ials_eval_set *e, int64_t n_rows, const int64_t *gt_indptr, const int32_t *gt_indices,
                        int gt_on_device, cudaStream_t s) {
  e->n_rows = n_rows;
  // ground truth: rows sorted ascending (a binary search per recommended item)
  int64_t gnnz = 0;
  e->gt_indptr.alloc(n_rows + 1);
  if (gt_on_device) {
    int64_t ends[2] = {0, 0};
    CUDA_CHECK(cudaMemcpyAsync(&ends[0], gt_indptr, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    CUDA_CHECK(cudaMemcpyAsync(&ends[1], gt_indptr + n_rows, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    CUDA_CHECK(cudaStreamSynchronize(s));
    require(ends[0] == 0 && ends[1] >= 0, "ground-truth indptr must start at 0");
    gnnz = ends[1];
    require(gnnz == 0 || gt_indices != nullptr, "ground-truth indices are null");
    CUDA_CHECK(cudaMemcpyAsync(e->gt_indptr.get(), gt_indptr, sizeof(int64_t) * (n_rows + 1),
                               cudaMemcpyDeviceToDevice, s));
    e->gt_indices.alloc(std::max<int64_t>(gnnz, 1));
    if (gnnz)
      CUDA_CHECK(cudaMemcpyAsync(e->gt_indices.get(), gt_indices, sizeof(int32_t) * gnnz,
                                 cudaMemcpyDeviceToDevice, s));
  } else {
    require(gt_indptr[0] == 0, "ground-truth indptr must start at 0");
    gnnz = gt_indptr[n_rows];
    require(gnnz == 0 || gt_indices != nullptr, "ground-truth indices are null");
    for (int64_t r = 0; r < n_rows; r++) {
      require(gt_indptr[r + 1] >= gt_indptr[r], "ground-truth indptr must be non-decreasing");
      for (int64_t j = gt_indptr[r] + 1; j < gt_indptr[r + 1]; j++)
        require(gt_indices[j - 1] <= gt_indices[j], "ground-truth rows must be sorted");
    }
    CUDA_CHECK(cudaMemcpyAsync(e->gt_indptr.get(), gt_indptr, sizeof(int64_t) * (n_rows + 1),
                               cudaMemcpyHostToDevice, s));
    e->gt_indices.alloc(std::max<int64_t>(gnnz, 1));
    if (gnnz)
      CUDA_CHECK(cudaMemcpyAsync(e->gt_indices.get(), gt_indices, sizeof(int32_t) * gnnz,
                                 cudaMemcpyHostToDevice, s));
  }
}

// The rest of a set, once its mask is staged: the allow-lists (they need the mask's sortedness), the
// discount tables, cutoffs and accumulators, on stream s
void stage_lists_and_accumulators(ials_trainer *t, ials_eval_set *e, int64_t allow_n_lists,
                                  const int64_t *allow_indptr, const int32_t *allow_indices, const int64_t *cutoffs,
                                  int64_t n_cutoffs, int64_t kmax, int recall_with_cutoff, cudaStream_t s) {
  e->device = t->device;
  e->n_items = t->I;
  e->n_cut = (int)n_cutoffs;
  e->kmax = kmax;
  e->recall_with_cutoff = recall_with_cutoff ? 1 : 0;
  if (allow_n_lists > 0) {
    if (!(score_topk_tc_supported(t->ld, kmax) && e->mask_sorted))
      throw NotImplemented("allow-lists need the fused tensor-core kernel (cutoff <= 128, sorted mask rows)");
    stage_allow_lists(t->I, allow_n_lists, allow_indptr, allow_indices, e->a_words, e->a_indptr, e->a_indices,
                      s, e->allow);
  }
  // prepare_dcg_discount (evaluator.cpp:42-48) and its prefix sums, the Evaluator's table
  std::vector<double> disc((size_t)kmax), cum((size_t)kmax);
  std::vector<int32_t> cut32((size_t)n_cutoffs);
  double run = 0;
  for (int64_t j = 0; j < kmax; j++) {
    disc[j] = 1.0 / std::log2(2.0 + (double)j);
    cum[j] = (run += disc[j]);
  }
  for (int64_t c = 0; c < n_cutoffs; c++) cut32[c] = (int32_t)cutoffs[c];
  CUDA_CHECK(cudaMemcpyAsync(e->discount.alloc(kmax), disc.data(), sizeof(double) * kmax, cudaMemcpyHostToDevice, s));
  CUDA_CHECK(cudaMemcpyAsync(e->cum.alloc(kmax), cum.data(), sizeof(double) * kmax, cudaMemcpyHostToDevice, s));
  CUDA_CHECK(cudaMemcpyAsync(e->cutoffs.alloc(n_cutoffs), cut32.data(), sizeof(int32_t) * n_cutoffs,
                             cudaMemcpyHostToDevice, s));
  e->sums.alloc(5 * n_cutoffs);
  e->counts.alloc(2 * n_cutoffs);
  e->hist.alloc(n_cutoffs * t->I);
  e->partial.alloc(5 * metrics_partials(kListSlabRows) * std::min<int64_t>(n_cutoffs, kMaxMetricsCutoffs));
  e->div_out.alloc(3);
  zero_accumulators(e, s);
}

// The list job of a pass: top-kmax with the set's mask and allow-lists into the trainer's list buffers
ListJob list_job(ials_trainer *t, const ials_eval_set *e, int64_t chunk) {
  ListJob job = e->allow;
  job.catalog = t->factor[1].get();
  job.n_catalog = t->I;
  job.k = e->kmax;
  job.mask_mode = e->mask_mode;
  job.m_indptr = e->m_indptr.get();
  job.m_indices = e->m_indices.get();
  job.mask_sorted = e->mask_sorted;
  job.idx = t->rec_idx.ensure(chunk * e->kmax);
  job.score = t->rec_score.ensure(chunk * e->kmax);
  job.count = t->rec_count.ensure(chunk);
  return job;
}

// Lists of `job` (produce_lists), then the metrics of every cutoff for its rows, set rows r0 + [0, job.rows)
void lists_and_metrics(ials_trainer *t, ials_eval_set *e, ListJob &job, int64_t r0) {
  job.m_row0 = r0;
  job.a_row0 = r0;
  produce_lists(t, job);
  for (int c0 = 0; c0 < e->n_cut; c0 += kMaxMetricsCutoffs) {
    const int nc = std::min(kMaxMetricsCutoffs, e->n_cut - c0);
    launch_metrics_rows(job.idx, job.count, job.rows, (int)e->kmax, e->gt_indptr.get() + r0, e->gt_indices.get(),
                        e->discount.get(), e->cum.get(), e->cutoffs.get() + c0, nc, e->recall_with_cutoff,
                        e->n_items, e->partial.get(), e->sums.get() + 5 * c0, e->counts.get() + c0,
                        e->counts.get() + e->n_cut + c0, e->hist.get() + (int64_t)c0 * e->n_items, t->stream);
  }
}

}  // namespace

extern "C" {

int ials_eval_set_create(ials_trainer *t, int64_t row_begin, int64_t n_rows, const int64_t *gt_indptr,
                         const int32_t *gt_indices, int gt_on_device, const int64_t *mask_indptr,
                         const int32_t *mask_indices, int64_t allow_n_lists, const int64_t *allow_indptr,
                         const int32_t *allow_indices, const int64_t *cutoffs, int64_t n_cutoffs,
                         int recall_with_cutoff, ials_eval_set **out) {
  return guarded([&] {
    require(t != nullptr && out != nullptr, "null pointer");
    *out = nullptr;
    require(row_begin >= 0 && n_rows >= 0 && row_begin + n_rows <= t->U, "bad user block");
    const int64_t kmax = check_cutoffs(t, cutoffs, n_cutoffs);
    require(gt_indptr != nullptr, "ground-truth indptr is null");
    require(allow_n_lists == 0 || allow_n_lists == 1 || allow_n_lists == n_rows,
            "allow-lists: one shared list or one per row");
    const bool custom_mask = mask_indptr != nullptr;
    if (!custom_mask) {
      if (!t->has_X) throw std::runtime_error("no training matrix to mask with");
      require(n_rows == 0 || (row_begin >= t->X.row_base && row_begin + n_rows <= t->X.row_base + t->X.n_rows),
              "mask='train' on a sharded trainer needs a user block inside the rank's shard");
    }
    DeviceGuard g(t->device);
    cudaStream_t s = t->stream;
    auto e = std::make_unique<ials_eval_set>();
    StreamSyncOnExit sync{s};  // the host staging below outlives the asynchronous copies
    e->row_begin = row_begin;
    stage_ground_truth(e.get(), n_rows, gt_indptr, gt_indices, gt_on_device, s);
    if (custom_mask) {  // stored zeros already removed, as scipy's .nonzero() does
      e->mask_mode = 2;
      stage_mask(n_rows, t->I, mask_indptr, mask_indices, e->m_indptr, e->m_indices, s);
      e->mask_sorted = mask_rows_sorted(n_rows, mask_indptr, mask_indices);
    } else {
      if (t->X.sorted_state < 0)
        t->X.sorted_state = csr_rows_strictly_sorted(t->X.indptr.get(), t->X.indices.get(), t->X.n_rows, s) ? 1 : 0;
      e->mask_sorted = t->X.sorted_state == 1;
    }
    stage_lists_and_accumulators(t, e.get(), allow_n_lists, allow_indptr, allow_indices, cutoffs, n_cutoffs, kmax,
                                 recall_with_cutoff, s);
    *out = e.release();
  });
}

int ials_eval_set_create_cold(ials_trainer *t, int64_t n_rows, int64_t n_cols, const int64_t *in_indptr,
                              const int32_t *in_indices, const float *in_data, const int64_t *gt_indptr,
                              const int32_t *gt_indices, int on_device, const int64_t *mask_indptr,
                              const int32_t *mask_indices, int64_t allow_n_lists, const int64_t *allow_indptr,
                              const int32_t *allow_indices, const int64_t *cutoffs, int64_t n_cutoffs,
                              int recall_with_cutoff, ials_eval_set **out) {
  return guarded([&] {
    require(t != nullptr && out != nullptr, "null pointer");
    *out = nullptr;
    require(n_rows >= 0 && n_cols >= 0, "negative shape");
    if (n_cols != t->I)  // Solver::X_to_vector, IALSTrainer.hpp:126-131
      throw InvalidArgument("Shape mismatch: X.cols() = " + std::to_string(n_cols) +
                            " but other.factor.rows() = " + std::to_string(t->I) + ".");
    require(n_rows < (1ll << 31), "cold users must fit int32");
    const int64_t kmax = check_cutoffs(t, cutoffs, n_cutoffs);
    require(in_indptr != nullptr && gt_indptr != nullptr, "indptr is null");
    require(allow_n_lists == 0 || allow_n_lists == 1 || allow_n_lists == n_rows,
            "allow-lists: one shared list or one per row");
    DeviceGuard g(t->device);
    cudaStream_t s = t->stream;
    // the input is validated, split into chunks and (by default) turned into the mask on the host;
    // device arrays are staged there once
    std::vector<int64_t> ip_host;
    std::vector<int32_t> ix_host;
    std::vector<float> dt_host;
    const int64_t *ip = in_indptr;
    const int32_t *ix = in_indices;
    const float *dt = in_data;
    if (on_device) {
      ip_host.resize((size_t)n_rows + 1);
      CUDA_CHECK(cudaMemcpy(ip_host.data(), in_indptr, sizeof(int64_t) * (n_rows + 1), cudaMemcpyDeviceToHost));
      const int64_t nnz = ip_host[(size_t)n_rows];
      require(ip_host[0] == 0 && nnz >= 0, "indptr[0] must be 0");
      require(nnz == 0 || (in_indices != nullptr && in_data != nullptr), "indices/data are null");
      ix_host.resize((size_t)nnz);
      dt_host.resize((size_t)nnz);
      if (nnz) {
        CUDA_CHECK(cudaMemcpy(ix_host.data(), in_indices, sizeof(int32_t) * nnz, cudaMemcpyDeviceToHost));
        CUDA_CHECK(cudaMemcpy(dt_host.data(), in_data, sizeof(float) * nnz, cudaMemcpyDeviceToHost));
      }
      ip = ip_host.data();
      ix = ix_host.data();
      dt = dt_host.data();
    }
    require(ip[0] == 0, "indptr[0] must be 0");
    for (int64_t r = 0; r < n_rows; r++) require(ip[r + 1] >= ip[r], "indptr must be non-decreasing");
    auto e = std::make_unique<ials_eval_set>();
    StreamSyncOnExit sync{s};  // the host staging below outlives the asynchronous copies
    e->cold = true;
    e->mask_mode = 2;
    const int64_t n_chunks = (n_rows + kListSlabRows - 1) / kListSlabRows;
    e->input = std::vector<DeviceCsr>((size_t)n_chunks);
    for (int64_t c = 0; c < n_chunks; c++) {  // each chunk a CSR from 0: the fold-in solves it as a whole
      const int64_t r0 = c * kListSlabRows, m = std::min(kListSlabRows, n_rows - r0);
      std::vector<int64_t> sub((size_t)m + 1);
      for (int64_t r = 0; r <= m; r++) sub[r] = ip[r0 + r] - ip[r0];
      upload_csr(e->input[c], m, n_cols, sub.data(), ix + ip[r0], dt + ip[r0]);
      plan_csr(t, e->input[c]);
    }
    stage_ground_truth(e.get(), n_rows, gt_indptr, gt_indices, on_device, s);
    if (mask_indptr != nullptr) {  // masked_interactions replaces the input (evaluator.py:574-577)
      stage_mask(n_rows, t->I, mask_indptr, mask_indices, e->m_indptr, e->m_indices, s);
      e->mask_sorted = mask_rows_sorted(n_rows, mask_indptr, mask_indices);
    } else {  // the input's non-zeros, rows sorted: scipy's .nonzero() drops stored zeros (evaluator.py:432)
      std::vector<int64_t> mi((size_t)n_rows + 1, 0);
      std::vector<int32_t> mx;
      mx.reserve((size_t)ip[n_rows]);
      for (int64_t r = 0; r < n_rows; r++) {
        for (int64_t j = ip[r]; j < ip[r + 1]; j++)
          if (dt[j] != 0.f) mx.push_back(ix[j]);
        std::sort(mx.begin() + mi[r], mx.end());
        mi[r + 1] = (int64_t)mx.size();
      }
      stage_mask(n_rows, t->I, mi.data(), mx.data(), e->m_indptr, e->m_indices, s);
      e->mask_sorted = mask_rows_sorted(n_rows, mi.data(), mx.data());
      CUDA_CHECK(cudaStreamSynchronize(s));  // mi / mx are staged from this scope
    }
    stage_lists_and_accumulators(t, e.get(), allow_n_lists, allow_indptr, allow_indices, cutoffs, n_cutoffs, kmax,
                                 recall_with_cutoff, s);
    e->slab.alloc(std::max<int64_t>(std::min(n_rows, kListSlabRows) * t->ld, 1));
    *out = e.release();
  });
}

void ials_eval_set_destroy(ials_eval_set *e) {
  if (e == nullptr) return;
  int prev = -1;
  cudaGetDevice(&prev);
  cudaSetDevice(e->device);
  delete e;
  if (prev >= 0) cudaSetDevice(prev);
}

int ials_eval_set_reset(ials_eval_set *e, void *cuda_stream) {
  return guarded([&] {
    require(e != nullptr, "evaluation set is null");
    DeviceGuard g(e->device);
    zero_accumulators(e, (cudaStream_t)cuda_stream);
  });
}

int ials_eval_set_buffers(ials_eval_set *e, double **sums, int64_t **counts, int64_t **hist, int64_t *n_cutoffs,
                          int64_t *n_items) {
  return guarded([&] {
    require(e && sums && counts && hist && n_cutoffs && n_items, "null pointer");
    *sums = e->sums.get();
    *counts = reinterpret_cast<int64_t *>(e->counts.get());
    *hist = reinterpret_cast<int64_t *>(e->hist.get());
    *n_cutoffs = e->n_cut;
    *n_items = e->n_items;
  });
}

int ials_eval_set_diversity(ials_eval_set *e, void *cuda_stream, double *out) {
  return guarded([&] {
    require(e != nullptr && out != nullptr, "null pointer");
    DeviceGuard g(e->device);
    cudaStream_t s = (cudaStream_t)cuda_stream;
    StreamSyncOnExit sync{s};
    for (int c = 0; c < e->n_cut; c++) {
      diversity_of_histogram(e->hist.get() + (int64_t)c * e->n_items, e->n_items, e->div_ws, e->div_out.get(), s);
      CUDA_CHECK(cudaMemcpyAsync(out + 3 * c, e->div_out.get(), sizeof(double) * 3, cudaMemcpyDeviceToHost, s));
      CUDA_CHECK(cudaStreamSynchronize(s));
    }
  });
}

int ials_trainer_evaluate(ials_trainer *t, ials_eval_set *e, int64_t user_begin, int64_t user_end) {
  return guarded([&] {
    require(t != nullptr && e != nullptr, "null pointer");
    require(!e->cold, "a cold evaluation set: use ials_trainer_evaluate_cold");
    require(e->device == t->device && e->n_items == t->I, "the evaluation set belongs to another model");
    require(user_begin >= e->row_begin && user_begin <= user_end && user_end <= e->row_begin + e->n_rows,
            "users outside the evaluation set's rows");
    const int64_t rows = user_end - user_begin;
    if (rows == 0) return;
    if (e->mask_mode == 0)
      require(user_begin >= t->X.row_base && user_end <= t->X.row_base + t->X.n_rows,
              "mask='train' on a sharded trainer needs a user block inside the rank's shard");
    DeviceGuard g(t->device);
    StreamSyncOnExit sync{t->stream};
    const int64_t chunk = std::min(rows, kListSlabRows);
    ListJob job = list_job(t, e, chunk);
    for (int64_t b = 0; b < rows; b += chunk) {
      job.user_rows = t->factor[0].get() + (user_begin + b) * t->ld;
      job.rows = std::min(chunk, rows - b);
      job.x_row0 = user_begin + b - t->X.row_base;
      lists_and_metrics(t, e, job, user_begin + b - e->row_begin);  // set row of the chunk
    }
  });
}

int ials_trainer_evaluate_cold(ials_trainer *t, ials_eval_set *e, const ials_solver_config *solver,
                               int64_t row_begin, int64_t row_end) {
  return guarded([&] {
    require(t != nullptr && e != nullptr, "null pointer");
    check_solver(solver);
    require(e->cold, "not a cold evaluation set: use ials_trainer_evaluate");
    require(e->device == t->device && e->n_items == t->I, "the evaluation set belongs to another model");
    require(0 <= row_begin && row_begin <= row_end && row_end <= e->n_rows, "rows outside the evaluation set's rows");
    if (row_begin == row_end) return;
    DeviceGuard g(t->device);
    StreamSyncOnExit sync{t->stream};
    NoProfiling quiet(t);  // phase marks belong to epochs
    gram_side(t, 0);       // prepare_p of the fold-in (IALSTrainer.hpp:793), over the full item replica
    ListJob job = list_job(t, e, std::min(row_end - row_begin, kListSlabRows));
    for (int64_t c = row_begin / kListSlabRows; c * kListSlabRows < row_end; c++) {
      // Solver::X_to_vector (:123-140): the chunk's rows from zero against the item factors
      const DeviceCsr &csr = e->input[c];
      const int64_t c0 = c * kListSlabRows;
      CUDA_CHECK(cudaMemsetAsync(e->slab.get(), 0, sizeof(float) * csr.n_rows * t->ld, t->stream));
      run_solver(t, make_args(t, 0, e->slab.get(), csr, solver), csr, solver, t->stream);
      const int64_t lo = std::max(row_begin, c0), hi = std::min(row_end, c0 + csr.n_rows);
      job.user_rows = e->slab.get() + (lo - c0) * t->ld;
      job.rows = hi - lo;
      lists_and_metrics(t, e, job, lo);
    }
    sync_and_check(t);  // solver failures, with the reference's messages
  });
}

}  // extern "C"
