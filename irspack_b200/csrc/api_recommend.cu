// Serving behind the C ABI: dense scores of a user block, recommendation lists (masks, allow-lists,
// users by index, fold-in embeddings), standalone top-k of host scores and the ranking metrics.
#include <algorithm>
#include <vector>

#include "trainer.cuh"

using namespace ials;

namespace {

float *ensure_score_buf(ials_trainer *t, size_t bytes) { return reinterpret_cast<float *>(t->score_buf.ensure(bytes)); }

// A host mask CSR (the items excluded from each row's list) either is absent (both pointers null) or
// has an indptr; its indices may be null only when it holds no entry.
void check_mask_pointers(int64_t rows, const int64_t *indptr, const int32_t *indices) {
  require(indptr != nullptr ? indices != nullptr || indptr[rows] == 0 : indices == nullptr,
          "mask indptr / indices must both be given");
}

// Copies the top-k lists of `rows` rows back to the host (out_score optional) and waits for them.
void download_lists(const int32_t *d_idx, const float *d_sc, const int32_t *d_cnt, int64_t rows, int64_t k,
                    int32_t *out_idx, float *out_score, int32_t *out_count, cudaStream_t s) {
  CUDA_CHECK(cudaMemcpyAsync(out_idx, d_idx, sizeof(int32_t) * rows * k, cudaMemcpyDeviceToHost, s));
  if (out_score) CUDA_CHECK(cudaMemcpyAsync(out_score, d_sc, sizeof(float) * rows * k, cudaMemcpyDeviceToHost, s));
  CUDA_CHECK(cudaMemcpyAsync(out_count, d_cnt, sizeof(int32_t) * rows, cudaMemcpyDeviceToHost, s));
  CUDA_CHECK(cudaStreamSynchronize(s));
}

}  // namespace

namespace ials {

void stage_mask(int64_t rows, int64_t n_cols, const int64_t *indptr, const int32_t *indices,
                DeviceBuffer<int64_t> &d_indptr, DeviceBuffer<int32_t> &d_indices, cudaStream_t s) {
  require(indptr != nullptr && indptr[0] == 0, "mask indptr must start at 0");
  check_mask_pointers(rows, indptr, indices);
  const int64_t nnz = indptr[rows];
  for (int64_t j = 0; j < nnz; j++) require(indices[j] >= 0 && indices[j] < n_cols, "mask index out of range");
  d_indptr.ensure(rows + 1);
  d_indices.ensure(std::max<int64_t>(nnz, 1));
  CUDA_CHECK(cudaMemcpyAsync(d_indptr.get(), indptr, sizeof(int64_t) * (rows + 1), cudaMemcpyHostToDevice, s));
  if (nnz)
    CUDA_CHECK(cudaMemcpyAsync(d_indices.get(), indices, sizeof(int32_t) * nnz, cudaMemcpyHostToDevice, s));
}

bool mask_rows_sorted(int64_t rows, const int64_t *indptr, const int32_t *indices) {
  for (int64_t r = 0; r < rows; r++)
    for (int64_t j = indptr[r] + 1; j < indptr[r + 1]; j++)
      if (indices[j - 1] >= indices[j]) return false;
  return true;
}

void stage_allow_lists(int64_t n_items, int64_t n_lists, const int64_t *indptr, const int32_t *indices,
                       std::vector<uint32_t> &words, DeviceBuffer<int64_t> &d_indptr,
                       DeviceBuffer<int32_t> &d_indices, cudaStream_t s, ListJob &job) {
  require(indptr != nullptr && indptr[0] == 0, "allow indptr must start at 0");
  const int64_t annz = indptr[n_lists];
  require(annz == 0 || indices != nullptr, "allow indices are null");
  for (int64_t r = 0; r < n_lists; r++)
    for (int64_t j = indptr[r]; j < indptr[r + 1]; j++) {
      require(indices[j] >= 0 && indices[j] < n_items, "allowed item out of range");
      require(j == indptr[r] || indices[j - 1] < indices[j], "allow-lists must be strictly ascending");
    }
  job.allow_n_lists = n_lists;
  if (n_lists == 1) {  // a shared list goes to the kernel as a bitmap of the catalogue
    words.assign((size_t)((n_items + 31) / 32), 0u);  // outlives the asynchronous copy
    for (int64_t j = 0; j < annz; j++) words[indices[j] >> 5] |= 1u << (indices[j] & 31);
    uint32_t *bitmap = reinterpret_cast<uint32_t *>(d_indices.ensure(words.size()));
    CUDA_CHECK(cudaMemcpyAsync(bitmap, words.data(), sizeof(uint32_t) * words.size(), cudaMemcpyHostToDevice, s));
    job.a_bitmap = bitmap;
  } else {
    int64_t *ip = d_indptr.ensure(n_lists + 1);
    int32_t *ix = d_indices.ensure(std::max<int64_t>(annz, 1));
    CUDA_CHECK(cudaMemcpyAsync(ip, indptr, sizeof(int64_t) * (n_lists + 1), cudaMemcpyHostToDevice, s));
    if (annz) CUDA_CHECK(cudaMemcpyAsync(ix, indices, sizeof(int32_t) * annz, cudaMemcpyHostToDevice, s));
    job.a_indptr = ip;
    job.a_indices = ix;
  }
}

void produce_lists(ials_trainer *t, const ListJob &j) {
  require(j.catalog != nullptr || j.n_catalog == 0, "list job without a catalogue");
  const bool fused = score_topk_tc_supported(t->ld, j.k) && j.mask_sorted;
  if (j.rowmap != nullptr && j.mask_mode == 0 && !fused)
    throw NotImplemented("mask='train' for users picked by index needs the fused tensor-core kernel");
  if (j.allow_n_lists > 0 && !fused)
    throw NotImplemented("allow-lists need the fused tensor-core kernel (cutoff <= 128, sorted mask rows)");
  const int64_t rows = j.rows, k = j.k, n = j.n_catalog;
  if (fused) {
    // scores + mask + top-k in one tcgen05 kernel; only candidate keys touch HBM
    for (int64_t b = 0; b < rows; b += kListSlabRows) {
      const int64_t m = std::min(kListSlabRows, rows - b);
      void *scratch = ensure_score_buf(t, score_tc_scratch_bytes(m, n, k));
      const int64_t *mip = nullptr;
      const int32_t *mix = nullptr;
      const float *mdt = nullptr;
      int64_t mrow0 = 0;
      const int64_t *mrowmap = nullptr;
      if (j.mask_mode == 0) {
        mip = t->X.indptr.get(); mix = t->X.indices.get(); mdt = t->X.data.get();
        mrow0 = j.x_row0 + b;
        if (j.rowmap) { mrowmap = j.rowmap + b; mrow0 = -t->X.row_base; }
      } else if (j.mask_mode == 2) {
        mip = j.m_indptr; mix = j.m_indices; mrow0 = j.m_row0 + b;
      }
      launch_score_topk_tc(j.user_rows + b * t->ld, m, j.catalog, n, t->ld, mip,
                           mix, mdt, mrow0, (int)k, scratch, j.idx + b * k, j.score + b * k,
                           j.count + b, t->stream, (int)std::min<int64_t>(j.allow_n_lists, 2), j.a_indptr,
                           j.a_indices, j.a_row0 + b, j.a_bitmap, mrowmap);
    }
    return;
  }
  const int64_t slab = std::max<int64_t>(1, std::min<int64_t>(rows, (1ll << 29) / (4 * n)));
  float *buf = ensure_score_buf(t, sizeof(float) * slab * n);
  for (int64_t b = 0; b < rows; b += slab) {
    const int64_t m = std::min(slab, rows - b);
    launch_scores(j.user_rows + b * t->ld, m, j.catalog, n, t->ld, buf, n, t->stream);
    if (j.mask_mode == 0)
      launch_mask_rows(buf, n, t->X.indptr.get(), t->X.indices.get(), t->X.data.get(), j.x_row0 + b, m, 0,
                       t->stream);
    else if (j.mask_mode == 2)
      launch_mask_rows(buf, n, j.m_indptr, j.m_indices, nullptr, j.m_row0 + b, m, 0, t->stream);
    launch_topk_rows(buf, n, m, n, (int)k, j.idx + b * k, j.score + b * k, j.count + b, t->stream);
  }
}

}  // namespace ials

namespace {

// The query rows and the mask of a list request, staged on the device into job.user_rows, rowmap,
// mask_mode, x_row0, m_indptr / m_indices and mask_sorted.  user_idx != nullptr: the rows are users
// user_idx[0 .. rows), gathered on the device; user_emb != nullptr: the rows are the host embeddings
// user_emb[rows x K] (fold-in results); otherwise users [begin, begin + rows).  Call under the trainer's
// device, with its stream synchronised on exit (the staging buffers stay with the trainer).
void stage_queries(ials_trainer *t, const int64_t *user_idx, const float *user_emb, int64_t begin,
                          int64_t rows, int mask_mode, const int64_t *mask_indptr, const int32_t *mask_indices,
                          ListJob &job) {
  if (mask_mode == 0 && !t->has_X) throw std::runtime_error("no training matrix to mask with");
  if (mask_mode == 0 && user_idx == nullptr && user_emb == nullptr)  // a sharded trainer only holds its own users' rows of X
    require(begin >= t->X.row_base && begin + rows <= t->X.row_base + t->X.n_rows,
            "mask='train' on a sharded trainer needs a user block inside the rank's shard");
  if (user_idx != nullptr)
    for (int64_t r = 0; r < rows; r++) {
      require(user_idx[r] >= 0 && user_idx[r] < t->U, "user index out of range");
      if (mask_mode == 0)
        require(user_idx[r] >= t->X.row_base && user_idx[r] < t->X.row_base + t->X.n_rows,
                "mask='train' on a sharded trainer needs users inside the rank's shard");
    }
  // the fused tensor-core kernel walks each mask row with a cursor: column ids must ascend
  job.mask_sorted = true;
  if (mask_mode == 0) {
    if (t->X.sorted_state < 0)
      t->X.sorted_state =
          csr_rows_strictly_sorted(t->X.indptr.get(), t->X.indices.get(), t->X.n_rows, t->stream) ? 1 : 0;
    job.mask_sorted = t->X.sorted_state == 1;
  }
  if (mask_mode == 2) {
    stage_mask(rows, t->I, mask_indptr, mask_indices, t->rec_mindptr, t->rec_mindices, t->stream);
    job.mask_sorted = mask_rows_sorted(rows, mask_indptr, mask_indices);
    job.m_indptr = t->rec_mindptr.get();
    job.m_indices = t->rec_mindices.get();
  }
  job.mask_mode = mask_mode;
  job.x_row0 = begin - t->X.row_base;
  job.user_rows = t->factor[0].get() + begin * t->ld;
  // users picked by index: their factor rows are gathered into a dense block first
  if (user_idx != nullptr) {
    int64_t *d_uidx = t->rec_uidx.ensure(rows);
    float *gathered = t->rec_users.ensure(rows * t->ld);
    CUDA_CHECK(cudaMemcpyAsync(d_uidx, user_idx, sizeof(int64_t) * rows, cudaMemcpyHostToDevice, t->stream));
    launch_gather_rows(t->factor[0].get(), t->ld, d_uidx, rows, gathered, t->stream);
    job.user_rows = gathered;
    job.rowmap = d_uidx;
  }
  if (user_emb != nullptr) {  // host embeddings [rows x K] -> padded device rows [rows x ld]
    float *staged = t->rec_emb.ensure(rows * t->K);
    float *padded = t->rec_users.ensure(rows * t->ld);
    CUDA_CHECK(cudaMemcpyAsync(staged, user_emb, sizeof(float) * rows * t->K, cudaMemcpyHostToDevice, t->stream));
    launch_pad_copy(staged, rows, (int)t->K, padded, t->ld, t->stream);
    job.user_rows = padded;
  }
}

// Validates host candidate lists: indptr from 0 and non-decreasing, item ids in [0, n_items), and
// strictly ascending inside each list when `strict` (lists that are ranked; scored pairs may repeat)
void check_candidates(int64_t n_items, int64_t n_lists, const int64_t *indptr, const int32_t *indices,
                             bool strict) {
  require(indptr != nullptr && indptr[0] == 0, "candidate indptr must start at 0");
  for (int64_t r = 0; r < n_lists; r++) require(indptr[r + 1] >= indptr[r], "candidate indptr must be non-decreasing");
  require(indptr[n_lists] == 0 || indices != nullptr, "candidate indices are null");
  for (int64_t r = 0; r < n_lists; r++)
    for (int64_t j = indptr[r]; j < indptr[r + 1]; j++) {
      require(indices[j] >= 0 && indices[j] < n_items, "candidate item out of range");
      require(!strict || j == indptr[r] || indices[j - 1] < indices[j], "candidate lists must be strictly ascending");
    }
}

// Uploads validated candidate lists into the trainer's grow-only list buffers; shared: list 0 serves
// every row
CandSegments stage_candidates(ials_trainer *t, int64_t n_lists, const int64_t *indptr,
                                     const int32_t *indices, bool shared) {
  const int64_t nnz = indptr[n_lists];
  int64_t *ip = t->rec_aindptr.ensure(n_lists + 1);
  int32_t *ix = t->rec_aindices.ensure(std::max<int64_t>(nnz, 1));
  CUDA_CHECK(cudaMemcpyAsync(ip, indptr, sizeof(int64_t) * (n_lists + 1), cudaMemcpyHostToDevice, t->stream));
  if (nnz) CUDA_CHECK(cudaMemcpyAsync(ix, indices, sizeof(int32_t) * nnz, cudaMemcpyHostToDevice, t->stream));
  return CandSegments{ip, ix, 0, 0, shared ? nnz : -1};
}

// Rows [b, b + m) of a call whose (row, candidate) pairs share one pass of the score scratch: at most
// kListSlabRows rows and, unless one row alone has more, kCandSlabPairs pairs.  tasks[r] (rows + 1
// entries): the first score task of row r, one per kCandChunk of its candidates (launch_cand_scores).
struct CandSlab {
  int64_t b, m, pairs, max_len;
};
constexpr int64_t kCandSlabPairs = 1ll << 26;  // 256 MB of FP32 scores
std::vector<CandSlab> plan_candidate_slabs(int64_t rows, const int64_t *indptr, bool shared,
                                           std::vector<int64_t> &tasks) {
  std::vector<CandSlab> slabs;
  tasks.assign((size_t)rows + 1, 0);
  for (int64_t r = 0; r < rows; r++) {
    const int64_t len = shared ? indptr[1] : indptr[r + 1] - indptr[r];
    tasks[r + 1] = tasks[r] + ceil_div(len, kCandChunk);
    if (slabs.empty() || slabs.back().m == kListSlabRows || slabs.back().pairs + len > kCandSlabPairs)
      slabs.push_back(CandSlab{r, 0, 0, 0});
    CandSlab &c = slabs.back();
    c.m++;
    c.pairs += len;
    c.max_len = std::max(c.max_len, len);
  }
  return slabs;
}

const int64_t *stage_candidate_tasks(ials_trainer *t, const std::vector<int64_t> &tasks) {
  int64_t *d = t->cand_tasks.ensure(tasks.size());
  CUDA_CHECK(cudaMemcpyAsync(d, tasks.data(), sizeof(int64_t) * tasks.size(), cudaMemcpyHostToDevice, t->stream));
  return d;
}

int64_t max_slab_pairs(const std::vector<CandSlab> &slabs) {
  int64_t n = 1;
  for (const CandSlab &c : slabs) n = std::max(n, c.pairs);
  return n;
}

// Checks common to the candidate entry points: the query form (user_idx / user_emb / [begin, end))
void check_query_form(const ials_trainer *t, const int64_t *user_idx, const float *user_emb, int64_t begin,
                             int64_t end) {
  require(t != nullptr, "trainer is null");
  require(user_idx == nullptr || user_emb == nullptr, "give users by index or embeddings, not both");
  require(end >= begin && begin >= 0 && (user_idx != nullptr || user_emb != nullptr ? begin == 0 : end <= t->U),
          "bad user block");
}

}  // namespace

extern "C" {

int ials_trainer_user_scores(ials_trainer *t, int64_t begin, int64_t end,
                             const ials_solver_config *solver, float *out_host) {
  return guarded([&] {
    require(t != nullptr, "trainer is null");
    require(solver != nullptr, "solver_config is null");
    // IALSTrainer.hpp:944-951
    require(solver->n_threads > 0, "n_threads must be strictly positive.");
    require(end >= begin, "userblock_end must be greater than or equal to userblock_begin");
    require(begin >= 0 && t->U >= end, "userblock_end must be smaller than or equal to n_users");
    const int64_t rows = end - begin;
    if (rows == 0 || t->I == 0) return;
    require(out_host != nullptr, "out is null");
    DeviceGuard g(t->device);
    // bound the device staging buffer; large blocks are produced in slabs
    const int64_t slab = std::max<int64_t>(1, std::min<int64_t>(rows, (1ll << 30) / (4 * t->I)));
    float *buf = ensure_score_buf(t, sizeof(float) * slab * t->I);
    for (int64_t b = 0; b < rows; b += slab) {
      const int64_t m = std::min(slab, rows - b);
      if (score_tc_supported(t->ld, 1))
        launch_scores_tc(t->factor[0].get() + (begin + b) * t->ld, m, t->factor[1].get(), t->I, t->ld, buf, t->I,
                         t->stream);
      else
        launch_scores(t->factor[0].get() + (begin + b) * t->ld, m, t->factor[1].get(), t->I, t->ld, buf, t->I,
                      t->stream);
      CUDA_CHECK(cudaMemcpyAsync(out_host + b * t->I, buf, sizeof(float) * m * t->I,
                                 cudaMemcpyDeviceToHost, t->stream));
      CUDA_CHECK(cudaStreamSynchronize(t->stream));
    }
  });
}
// user_idx != nullptr: the rows are users user_idx[0 .. end) (begin = 0), gathered on the device;
// user_emb != nullptr: the rows are the host embeddings user_emb[end x K] (begin = 0; fold-in results)
static int recommend_impl(ials_trainer *t, const int64_t *user_idx, const float *user_emb, int64_t begin,
                          int64_t end, int64_t k, int mask_mode,
                          const int64_t *mask_indptr, const int32_t *mask_indices, int64_t allow_n_lists,
                          const int64_t *allow_indptr, const int32_t *allow_indices,
                          int32_t *out_idx, float *out_score, int32_t *out_count) {
  return guarded([&] {
    require(t != nullptr, "trainer is null");
    require(end >= begin && begin >= 0 && (user_idx != nullptr || user_emb != nullptr || end <= t->U),
            "bad user block");
    require(user_emb == nullptr || mask_mode != 0, "embeddings have no training rows: give the mask explicitly");
    require(k >= 1 && k <= t->I, "cutoff must be in [1, n_items]");  // evaluator.cpp:265-266
    require(k <= 1024, "k > 1024 is not supported");
    require(mask_mode >= 0 && mask_mode <= 2, "mask_mode must be 0, 1 or 2");
    const int64_t rows = end - begin;
    if (rows == 0) return;
    require(out_idx != nullptr && out_count != nullptr, "output pointer is null");
    DeviceGuard g(t->device);
    StreamSyncOnExit sync{t->stream};  // the staging buffers stay with the trainer
    ListJob job;
    stage_queries(t, user_idx, user_emb, begin, rows, mask_mode, mask_indptr, mask_indices, job);
    int32_t *d_idx = t->rec_idx.ensure(rows * k);
    float *d_sc = t->rec_score.ensure(rows * k);
    int32_t *d_cnt = t->rec_count.ensure(rows);
    job.catalog = t->factor[1].get();
    job.n_catalog = t->I;
    job.rows = rows;
    job.k = k;
    job.idx = d_idx;
    job.score = d_sc;
    job.count = d_cnt;
    if (allow_n_lists > 0) {
      require(allow_n_lists == 1 || allow_n_lists == rows, "allow-lists: one shared list or one per row");
      stage_allow_lists(t->I, allow_n_lists, allow_indptr, allow_indices, t->rec_abitmap_host, t->rec_aindptr,
                        t->rec_aindices, t->stream, job);
    }
    produce_lists(t, job);
    download_lists(d_idx, d_sc, d_cnt, rows, k, out_idx, out_score, out_count, t->stream);
  });
}

int ials_trainer_recommend(ials_trainer *t, int64_t begin, int64_t end, int64_t k, int mask_mode,
                           const int64_t *mask_indptr, const int32_t *mask_indices,
                           int32_t *out_idx, float *out_score, int32_t *out_count) {
  return recommend_impl(t, nullptr, nullptr, begin, end, k, mask_mode, mask_indptr, mask_indices, 0, nullptr,
                        nullptr, out_idx, out_score, out_count);
}

int ials_trainer_recommend_allowed(ials_trainer *t, int64_t begin, int64_t end, int64_t k, int mask_mode,
                                   const int64_t *mask_indptr, const int32_t *mask_indices, int64_t allow_n_lists,
                                   const int64_t *allow_indptr, const int32_t *allow_indices, int32_t *out_idx,
                                   float *out_score, int32_t *out_count) {
  return recommend_impl(t, nullptr, nullptr, begin, end, k, mask_mode, mask_indptr, mask_indices, allow_n_lists,
                        allow_indptr, allow_indices, out_idx, out_score, out_count);
}

int ials_trainer_recommend_users(ials_trainer *t, const int64_t *user_indices, int64_t n_users, int64_t k,
                                 int mask_mode, const int64_t *mask_indptr, const int32_t *mask_indices,
                                 int64_t allow_n_lists, const int64_t *allow_indptr, const int32_t *allow_indices,
                                 int32_t *out_idx, float *out_score, int32_t *out_count) {
  if (n_users > 0 && user_indices == nullptr) return guarded([] { require(false, "user_indices is null"); });
  static const int64_t none = 0;
  return recommend_impl(t, user_indices ? user_indices : &none, nullptr, 0, n_users, k, mask_mode, mask_indptr,
                        mask_indices, allow_n_lists, allow_indptr, allow_indices, out_idx, out_score, out_count);
}

int ials_trainer_recommend_embeddings(ials_trainer *t, const float *user_embeddings, int64_t n_rows, int64_t k,
                                      int mask_mode, const int64_t *mask_indptr, const int32_t *mask_indices,
                                      int64_t allow_n_lists, const int64_t *allow_indptr,
                                      const int32_t *allow_indices, int32_t *out_idx, float *out_score,
                                      int32_t *out_count) {
  if (n_rows > 0 && user_embeddings == nullptr) return guarded([] { require(false, "user_embeddings is null"); });
  static const float none = 0.f;
  return recommend_impl(t, nullptr, user_embeddings ? user_embeddings : &none, 0, n_rows, k, mask_mode,
                        mask_indptr, mask_indices, allow_n_lists, allow_indptr, allow_indices, out_idx, out_score,
                        out_count);
}

int ials_trainer_similar(ials_trainer *t, int side, const int64_t *query_idx, int64_t begin, int64_t end,
                         int64_t k, int metric, int exclude_self, const int64_t *forbid_indptr,
                         const int32_t *forbid_indices, int64_t allow_n_lists, const int64_t *allow_indptr,
                         const int32_t *allow_indices, int32_t *out_idx, float *out_score, int32_t *out_count) {
  return guarded([&] {
    require(t != nullptr, "trainer is null");
    require_side(side);
    const int64_t n = t->n_rows(side);
    require(end >= begin && begin >= 0 && (query_idx != nullptr ? begin == 0 : end <= n), "bad query block");
    require(metric == IALS_SIMILARITY_DOT || metric == IALS_SIMILARITY_COSINE, "metric must be 'cosine' or 'dot'");
    require(k >= 1 && k <= n, "cutoff must be in [1, rows of the side]");
    require(k <= 1024, "k > 1024 is not supported");
    const int64_t rows = end - begin;
    if (rows == 0) return;
    require(out_idx != nullptr && out_count != nullptr, "output pointer is null");
    if (query_idx != nullptr)
      for (int64_t r = 0; r < rows; r++) require(query_idx[r] >= 0 && query_idx[r] < n, "query index out of range");
    const bool forbid = forbid_indptr != nullptr;
    if (forbid) {
      require(forbid_indptr[0] == 0, "forbidden indptr must start at 0");
      for (int64_t r = 0; r < rows; r++)
        require(forbid_indptr[r + 1] >= forbid_indptr[r], "forbidden indptr must be non-decreasing");
    }
    check_mask_pointers(rows, forbid_indptr, forbid_indices);
    if (allow_n_lists > 0)
      require(allow_n_lists == 1 || allow_n_lists == rows, "allow-lists: one shared list or one per query");
    DeviceGuard g(t->device);
    // the mask: row r hides the query itself and its forbidden rows, strictly ascending (the fused
    // kernel's cursor).  A range of queries without forbidden lists reads row begin + r of a CSR built
    // on the device; otherwise the rows are merged here, one per query.
    std::vector<int64_t> m_indptr;
    std::vector<int32_t> m_indices;
    StreamSyncOnExit sync{t->stream};  // the staging buffers stay with the trainer
    ListJob job;
    job.mask_mode = 1;
    int64_t m_base = 0;
    if (forbid || (exclude_self && query_idx != nullptr)) {
      m_indptr.assign((size_t)rows + 1, 0);
      m_indices.reserve((size_t)((forbid ? forbid_indptr[rows] : 0) + (exclude_self ? rows : 0)));
      for (int64_t r = 0; r < rows; r++) {
        const size_t first = m_indices.size();
        if (forbid)
          for (int64_t j = forbid_indptr[r]; j < forbid_indptr[r + 1]; j++) {
            require(forbid_indices[j] >= 0 && forbid_indices[j] < n, "forbidden index out of range");
            m_indices.push_back(forbid_indices[j]);
          }
        if (exclude_self) m_indices.push_back((int32_t)(query_idx != nullptr ? query_idx[r] : begin + r));
        std::sort(m_indices.begin() + first, m_indices.end());
        m_indices.erase(std::unique(m_indices.begin() + first, m_indices.end()), m_indices.end());
        m_indptr[r + 1] = (int64_t)m_indices.size();
      }
      stage_mask(rows, n, m_indptr.data(), m_indices.data(), t->rec_mindptr, t->rec_mindices, t->stream);
      job.mask_mode = 2;
      job.m_indptr = t->rec_mindptr.get();
      job.m_indices = t->rec_mindices.get();
    } else if (exclude_self) {
      int64_t *ip = t->sim_self_indptr.ensure(n + 1);
      int32_t *ix = t->sim_self_indices.ensure(n);
      launch_self_mask(ip, ix, n, t->stream);
      job.mask_mode = 2;
      job.m_indptr = ip;
      job.m_indices = ix;
      m_base = begin;
    }
    if (allow_n_lists > 0)
      stage_allow_lists(n, allow_n_lists, allow_indptr, allow_indices, t->rec_abitmap_host, t->rec_aindptr,
                        t->rec_aindices, t->stream, job);
    // cosine: the same product on a copy of the side scaled to unit norm, queries included
    const float *Y = t->factor[side].get();
    if (metric == IALS_SIMILARITY_COSINE) {
      float *unit = t->sim_norm.ensure(n * t->ld);
      launch_normalize_rows(Y, n, t->ld, unit, t->stream);
      Y = unit;
    }
    job.catalog = Y;
    job.n_catalog = n;
    const float *queries = Y + begin * t->ld;
    if (query_idx != nullptr) {
      int64_t *d_q = t->rec_uidx.ensure(rows);
      float *gathered = t->rec_users.ensure(rows * t->ld);
      CUDA_CHECK(cudaMemcpyAsync(d_q, query_idx, sizeof(int64_t) * rows, cudaMemcpyHostToDevice, t->stream));
      launch_gather_rows(Y, t->ld, d_q, rows, gathered, t->stream);
      queries = gathered;
    }
    // slabs of queries: the list buffers stay bounded and each slab's lists go to the host behind it
    const int64_t slab = std::min(rows, kListSlabRows);
    job.k = k;
    job.idx = t->rec_idx.ensure(slab * k);
    job.score = t->rec_score.ensure(slab * k);
    job.count = t->rec_count.ensure(slab);
    for (int64_t b = 0; b < rows; b += slab) {
      const int64_t m = std::min(slab, rows - b);
      job.user_rows = queries + b * t->ld;
      job.rows = m;
      job.m_row0 = m_base + b;
      job.a_row0 = b;
      produce_lists(t, job);
      CUDA_CHECK(cudaMemcpyAsync(out_idx + b * k, job.idx, sizeof(int32_t) * m * k, cudaMemcpyDeviceToHost,
                                 t->stream));
      if (out_score)
        CUDA_CHECK(cudaMemcpyAsync(out_score + b * k, job.score, sizeof(float) * m * k, cudaMemcpyDeviceToHost,
                                   t->stream));
      CUDA_CHECK(cudaMemcpyAsync(out_count + b, job.count, sizeof(int32_t) * m, cudaMemcpyDeviceToHost, t->stream));
    }
    CUDA_CHECK(cudaStreamSynchronize(t->stream));
  });
}

int ials_trainer_rank_candidates(ials_trainer *t, const int64_t *user_idx, const float *user_emb, int64_t begin,
                                 int64_t end, int64_t k, int mask_mode, const int64_t *mask_indptr,
                                 const int32_t *mask_indices, int64_t cand_n_lists, const int64_t *cand_indptr,
                                 const int32_t *cand_indices, int32_t *out_idx, float *out_score,
                                 int32_t *out_count) {
  return guarded([&] {
    check_query_form(t, user_idx, user_emb, begin, end);
    require(user_emb == nullptr || mask_mode != 0, "embeddings have no training rows: give the mask explicitly");
    require(k >= 1 && k <= t->I, "cutoff must be in [1, n_items]");
    require(k <= 1024, "k > 1024 is not supported");
    require(mask_mode >= 0 && mask_mode <= 2, "mask_mode must be 0, 1 or 2");
    const int64_t rows = end - begin;
    require(cand_n_lists == 1 || cand_n_lists == rows, "candidates: one shared list or one per row");
    check_candidates(t->I, cand_n_lists, cand_indptr, cand_indices, true);
    if (rows == 0) return;
    require(out_idx != nullptr && out_count != nullptr, "output pointer is null");
    DeviceGuard g(t->device);
    StreamSyncOnExit sync{t->stream};  // the staging buffers stay with the trainer
    ListJob job;
    stage_queries(t, user_idx, user_emb, begin, rows, mask_mode, mask_indptr, mask_indices, job);
    const bool shared = cand_n_lists == 1;
    const CandSegments lists = stage_candidates(t, cand_n_lists, cand_indptr, cand_indices, shared);
    CandMask mask;
    mask.sorted = job.mask_sorted;
    if (mask_mode == 0) {
      mask.indptr = t->X.indptr.get();
      mask.indices = t->X.indices.get();
      mask.data = t->X.data.get();
    } else if (mask_mode == 2) {
      mask.indptr = job.m_indptr;
      mask.indices = job.m_indices;
    }
    std::vector<int64_t> tasks;
    const std::vector<CandSlab> slabs = plan_candidate_slabs(rows, cand_indptr, shared, tasks);
    const int64_t *d_tasks = stage_candidate_tasks(t, tasks);
    float *scratch = ensure_score_buf(t, sizeof(float) * max_slab_pairs(slabs));
    const int64_t slab_rows = std::min(rows, kListSlabRows);
    int32_t *d_idx = t->rec_idx.ensure(slab_rows * k);
    float *d_sc = t->rec_score.ensure(slab_rows * k);
    int32_t *d_cnt = t->rec_count.ensure(slab_rows);
    for (const CandSlab &c : slabs) {
      CandSegments seg = lists;
      if (!shared) { seg.row0 = c.b; seg.base = cand_indptr[c.b]; }
      CandMask m = mask;
      if (mask_mode == 0 && job.rowmap != nullptr) { m.rowmap = job.rowmap + c.b; m.row0 = -t->X.row_base; }
      else if (mask_mode == 0) m.row0 = job.x_row0 + c.b;
      else if (mask_mode == 2) m.row0 = c.b;
      launch_cand_scores(job.user_rows + c.b * t->ld, c.m, t->ld, t->factor[1].get(), seg, d_tasks + c.b,
                         tasks[c.b + c.m] - tasks[c.b], m, scratch, t->stream);
      launch_topk_segments(scratch, seg, c.m, c.max_len, (int)k, d_idx, d_sc, d_cnt, t->stream);
      CUDA_CHECK(cudaMemcpyAsync(out_idx + c.b * k, d_idx, sizeof(int32_t) * c.m * k, cudaMemcpyDeviceToHost,
                                 t->stream));
      if (out_score)
        CUDA_CHECK(cudaMemcpyAsync(out_score + c.b * k, d_sc, sizeof(float) * c.m * k, cudaMemcpyDeviceToHost,
                                   t->stream));
      CUDA_CHECK(cudaMemcpyAsync(out_count + c.b, d_cnt, sizeof(int32_t) * c.m, cudaMemcpyDeviceToHost, t->stream));
    }
    CUDA_CHECK(cudaStreamSynchronize(t->stream));
  });
}

int ials_trainer_candidate_scores(ials_trainer *t, const int64_t *user_idx, const float *user_emb, int64_t begin,
                                  int64_t end, const int64_t *cand_indptr, const int32_t *cand_indices,
                                  float *out_scores) {
  return guarded([&] {
    check_query_form(t, user_idx, user_emb, begin, end);
    const int64_t rows = end - begin;
    check_candidates(t->I, rows, cand_indptr, cand_indices, false);
    if (rows == 0 || cand_indptr[rows] == 0) return;
    require(out_scores != nullptr, "output pointer is null");
    DeviceGuard g(t->device);
    StreamSyncOnExit sync{t->stream};  // the staging buffers stay with the trainer
    ListJob job;
    stage_queries(t, user_idx, user_emb, begin, rows, 1, nullptr, nullptr, job);
    const CandSegments lists = stage_candidates(t, rows, cand_indptr, cand_indices, false);
    std::vector<int64_t> tasks;
    const std::vector<CandSlab> slabs = plan_candidate_slabs(rows, cand_indptr, false, tasks);
    const int64_t *d_tasks = stage_candidate_tasks(t, tasks);
    float *scratch = ensure_score_buf(t, sizeof(float) * max_slab_pairs(slabs));
    for (const CandSlab &c : slabs) {
      CandSegments seg = lists;
      seg.row0 = c.b;
      seg.base = cand_indptr[c.b];
      launch_cand_scores(job.user_rows + c.b * t->ld, c.m, t->ld, t->factor[1].get(), seg, d_tasks + c.b,
                         tasks[c.b + c.m] - tasks[c.b], CandMask{}, scratch, t->stream);
      if (c.pairs)
        CUDA_CHECK(cudaMemcpyAsync(out_scores + seg.base, scratch, sizeof(float) * c.pairs, cudaMemcpyDeviceToHost,
                                   t->stream));
    }
    CUDA_CHECK(cudaStreamSynchronize(t->stream));
  });
}

int ials_metrics_accumulate(const int32_t *rec, const int32_t *count, int64_t rows, int64_t k,
                            const int64_t *gt_indptr, const int32_t *gt_indices, int64_t n_items,
                            int recall_with_cutoff, const double *discount, int device, void *cuda_stream,
                            double *acc, int64_t *valid_user, int64_t *item_cnt) {
  return guarded([&] {
    require(rows >= 0 && k >= 1 && n_items >= 1, "bad shape");
    if (rows == 0) return;
    require(rec && count && gt_indptr && discount && acc && valid_user && item_cnt, "null pointer");
    require(gt_indptr[0] == 0, "ground-truth indptr must start at 0");
    const int64_t gnnz = gt_indptr[rows];
    require(gnnz == 0 || gt_indices != nullptr, "ground-truth indices are null");
    for (int64_t r = 0; r < rows; r++) {
      require(gt_indptr[r + 1] >= gt_indptr[r], "ground-truth indptr must be non-decreasing");
      for (int64_t j = gt_indptr[r] + 1; j < gt_indptr[r + 1]; j++)
        require(gt_indices[j - 1] <= gt_indices[j], "ground-truth rows must be sorted");
    }
    for (int64_t j = 0; j < rows * k; j++) require(rec[j] >= -1 && rec[j] < n_items, "recommended item out of range");
    require_device(device);
    DeviceGuard g(device);
    cudaStream_t s = (cudaStream_t)cuda_stream;
    std::vector<double> cum((size_t)k);
    double run = 0;
    for (int64_t j = 0; j < k; j++) cum[j] = (run += discount[j]);
    // one allocation: rec | count | gt indptr | gt indices | discount | cum | cutoff | partials |
    // acc[5] | valid | total | item_cnt
    const int32_t cutoff = (int32_t)k;
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; };
    const size_t o_rec = take(sizeof(int32_t) * rows * k), o_cnt = take(sizeof(int32_t) * rows),
                 o_ip = take(sizeof(int64_t) * (rows + 1)), o_ix = take(sizeof(int32_t) * std::max<int64_t>(gnnz, 1)),
                 o_d = take(sizeof(double) * k), o_c = take(sizeof(double) * k), o_k = take(sizeof(int32_t)),
                 o_p = take(sizeof(double) * 5 * metrics_partials(rows)), o_acc = take(sizeof(double) * 5),
                 o_v = take(sizeof(unsigned long long)), o_t = take(sizeof(unsigned long long)),
                 o_ic = take(sizeof(unsigned long long) * n_items);
    DeviceBuffer<char> buf;
    StreamSyncOnExit sync{s};
    char *d = buf.alloc(off);
    CUDA_CHECK(cudaMemcpyAsync(d + o_rec, rec, sizeof(int32_t) * rows * k, cudaMemcpyHostToDevice, s));
    CUDA_CHECK(cudaMemcpyAsync(d + o_cnt, count, sizeof(int32_t) * rows, cudaMemcpyHostToDevice, s));
    CUDA_CHECK(cudaMemcpyAsync(d + o_ip, gt_indptr, sizeof(int64_t) * (rows + 1), cudaMemcpyHostToDevice, s));
    if (gnnz) CUDA_CHECK(cudaMemcpyAsync(d + o_ix, gt_indices, sizeof(int32_t) * gnnz, cudaMemcpyHostToDevice, s));
    CUDA_CHECK(cudaMemcpyAsync(d + o_d, discount, sizeof(double) * k, cudaMemcpyHostToDevice, s));
    CUDA_CHECK(cudaMemcpyAsync(d + o_c, cum.data(), sizeof(double) * k, cudaMemcpyHostToDevice, s));
    CUDA_CHECK(cudaMemcpyAsync(d + o_k, &cutoff, sizeof(int32_t), cudaMemcpyHostToDevice, s));
    CUDA_CHECK(cudaMemsetAsync(d + o_acc, 0, off - o_acc, s));
    launch_metrics_rows(reinterpret_cast<int32_t *>(d + o_rec), reinterpret_cast<int32_t *>(d + o_cnt), rows, (int)k,
                        reinterpret_cast<int64_t *>(d + o_ip), reinterpret_cast<int32_t *>(d + o_ix),
                        reinterpret_cast<double *>(d + o_d), reinterpret_cast<double *>(d + o_c),
                        reinterpret_cast<int32_t *>(d + o_k), 1, recall_with_cutoff, n_items,
                        reinterpret_cast<double *>(d + o_p), reinterpret_cast<double *>(d + o_acc),
                        reinterpret_cast<unsigned long long *>(d + o_v), reinterpret_cast<unsigned long long *>(d + o_t),
                        reinterpret_cast<unsigned long long *>(d + o_ic), s);
    double h_acc[5];
    unsigned long long h_valid = 0;
    std::vector<unsigned long long> h_cnt((size_t)n_items);
    CUDA_CHECK(cudaMemcpyAsync(h_acc, d + o_acc, sizeof(h_acc), cudaMemcpyDeviceToHost, s));
    CUDA_CHECK(cudaMemcpyAsync(&h_valid, d + o_v, sizeof(h_valid), cudaMemcpyDeviceToHost, s));
    CUDA_CHECK(cudaMemcpyAsync(h_cnt.data(), d + o_ic, sizeof(unsigned long long) * n_items, cudaMemcpyDeviceToHost, s));
    CUDA_CHECK(cudaStreamSynchronize(s));
    for (int i = 0; i < 5; i++) acc[i] += h_acc[i];
    *valid_user += (int64_t)h_valid;
    for (int64_t i = 0; i < n_items; i++) item_cnt[i] += (int64_t)h_cnt[i];
  });
}

int ials_topk_scores(const float *scores_host, int64_t rows, int64_t n_items, int64_t k,
                     const int64_t *mask_indptr, const int32_t *mask_indices, int device,
                     void *cuda_stream, int32_t *out_idx, float *out_score, int32_t *out_count) {
  return guarded([&] {
    require(rows >= 0 && n_items >= 0, "negative shape");
    require(k >= 1 && k <= n_items, "cutoff must be in [1, n_items]");
    require(k <= 1024, "k > 1024 is not supported");
    if (rows == 0) return;
    require(scores_host && out_idx && out_count, "null pointer");
    check_mask_pointers(rows, mask_indptr, mask_indices);
    require_device(device);
    DeviceGuard g(device);
    cudaStream_t s = (cudaStream_t)cuda_stream;
    DeviceBuffer<float> d_scores, d_sc;
    DeviceBuffer<int64_t> d_mindptr;
    DeviceBuffer<int32_t> d_mindices, d_idx, d_cnt;
    StreamSyncOnExit sync{s};
    const int64_t slab = std::max<int64_t>(1, std::min<int64_t>(rows, (1ll << 29) / (4 * n_items)));
    d_scores.alloc(slab * n_items);
    d_idx.alloc(rows * k);
    d_sc.alloc(rows * k);
    d_cnt.alloc(rows);
    if (mask_indptr) stage_mask(rows, n_items, mask_indptr, mask_indices, d_mindptr, d_mindices, s);
    for (int64_t b = 0; b < rows; b += slab) {
      const int64_t m = std::min(slab, rows - b);
      CUDA_CHECK(cudaMemcpyAsync(d_scores.get(), scores_host + b * n_items, sizeof(float) * m * n_items,
                                 cudaMemcpyHostToDevice, s));
      if (mask_indptr)
        launch_mask_rows(d_scores.get(), n_items, d_mindptr.get(), d_mindices.get(), nullptr, b, m, 0, s);
      launch_topk_rows(d_scores.get(), n_items, m, n_items, (int)k, d_idx.get() + b * k, d_sc.get() + b * k,
                       d_cnt.get() + b, s);
    }
    download_lists(d_idx.get(), d_sc.get(), d_cnt.get(), rows, k, out_idx, out_score, out_count, s);
  });
}

int ials_retrieve_recommend(const float *scores_host, int64_t rows, int64_t n_items, int64_t cutoff,
                            int64_t n_allowed_lists, const int64_t *allowed_indptr,
                            const int64_t *allowed_indices, int device, void *cuda_stream,
                            int32_t *out_idx, float *out_score, int32_t *out_count) {
  return guarded([&] {
    require(rows >= 0 && n_items >= 0 && cutoff >= 0, "negative shape");
    require(n_allowed_lists == 0 || n_allowed_lists == 1 || n_allowed_lists == rows,
            "allowed_indices, if not empty, must have a size equal to X.rows()");  // util.hpp:436-439
    const int64_t k = std::min(cutoff, n_items);
    if (k > 1024) throw NotImplemented("retrieve_recommend: cutoff > 1024 is not supported");
    require(rows == 0 || out_count != nullptr, "null pointer");
    if (rows == 0 || k == 0) {
      for (int64_t r = 0; r < rows; r++) out_count[r] = 0;
      return;
    }
    require(scores_host && out_idx && out_count, "null pointer");
    require(n_allowed_lists == 0 || allowed_indptr != nullptr, "null allowed_indptr");
    require_device(device);
    DeviceGuard g(device);
    cudaStream_t s = (cudaStream_t)cuda_stream;
    DeviceBuffer<float> d_scores, d_allowed, d_sc;
    DeviceBuffer<int64_t> d_aindptr, d_aindices;
    DeviceBuffer<int32_t> d_idx, d_cnt;
    StreamSyncOnExit sync{s};
    const int64_t slab = std::max<int64_t>(1, std::min<int64_t>(rows, (1ll << 29) / (4 * n_items)));
    d_scores.alloc(slab * n_items);
    d_idx.alloc(rows * k);
    d_sc.alloc(rows * k);
    d_cnt.alloc(rows);
    if (n_allowed_lists > 0) {
      require(allowed_indptr[0] == 0, "allowed indptr must start at 0");
      const int64_t annz = allowed_indptr[n_allowed_lists];
      require(annz == 0 || allowed_indices != nullptr, "null allowed_indices");
      d_allowed.alloc(slab * n_items);
      d_aindptr.alloc(n_allowed_lists + 1);
      d_aindices.alloc(std::max<int64_t>(annz, 1));
      CUDA_CHECK(cudaMemcpyAsync(d_aindptr.get(), allowed_indptr, sizeof(int64_t) * (n_allowed_lists + 1),
                                 cudaMemcpyHostToDevice, s));
      if (annz)
        CUDA_CHECK(cudaMemcpyAsync(d_aindices.get(), allowed_indices, sizeof(int64_t) * annz,
                                   cudaMemcpyHostToDevice, s));
    }
    for (int64_t b = 0; b < rows; b += slab) {
      const int64_t m = std::min(slab, rows - b);
      CUDA_CHECK(cudaMemcpyAsync(d_scores.get(), scores_host + b * n_items, sizeof(float) * m * n_items,
                                 cudaMemcpyHostToDevice, s));
      const float *cand = d_scores.get();
      if (d_allowed.get()) {
        launch_allow_rows(d_scores.get(), d_allowed.get(), n_items, d_aindptr.get(), d_aindices.get(),
                          n_allowed_lists, b, m, n_items, s);
        cand = d_allowed.get();
      }
      launch_topk_rows(cand, n_items, m, n_items, (int)k, d_idx.get() + b * k, d_sc.get() + b * k,
                       d_cnt.get() + b, s);
    }
    download_lists(d_idx.get(), d_sc.get(), d_cnt.get(), rows, k, out_idx, out_score, out_count, s);
  });
}
}  // extern "C"
