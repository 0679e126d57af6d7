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

// Validates a host mask CSR of `rows` rows over n_cols items and copies it into d_indptr / d_indices
// (grown as needed) on stream s.
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

// Copies the top-k lists of `rows` rows back to the host (out_score optional) and waits for them.
void download_lists(const int32_t *d_idx, const float *d_sc, const int32_t *d_cnt, int64_t rows, int64_t k,
                    int32_t *out_idx, float *out_score, int32_t *out_count, cudaStream_t s) {
  CUDA_CHECK(cudaMemcpyAsync(out_idx, d_idx, sizeof(int32_t) * rows * k, cudaMemcpyDeviceToHost, s));
  if (out_score) CUDA_CHECK(cudaMemcpyAsync(out_score, d_sc, sizeof(float) * rows * k, cudaMemcpyDeviceToHost, s));
  CUDA_CHECK(cudaMemcpyAsync(out_count, d_cnt, sizeof(int32_t) * rows, cudaMemcpyDeviceToHost, s));
  CUDA_CHECK(cudaStreamSynchronize(s));
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
    if (mask_mode == 0 && !t->has_X) throw std::runtime_error("no training matrix to mask with");
    if (mask_mode == 0 && user_idx == nullptr && user_emb == nullptr)  // a sharded trainer only holds its own users' rows of X
      require(begin >= t->X.row_base && end <= t->X.row_base + t->X.n_rows,
              "mask='train' on a sharded trainer needs a user block inside the rank's shard");
    if (user_idx != nullptr)
      for (int64_t r = 0; r < rows; r++) {
        require(user_idx[r] >= 0 && user_idx[r] < t->U, "user index out of range");
        if (mask_mode == 0)
          require(user_idx[r] >= t->X.row_base && user_idx[r] < t->X.row_base + t->X.n_rows,
                  "mask='train' on a sharded trainer needs users inside the rank's shard");
      }
    DeviceGuard g(t->device);
    StreamSyncOnExit sync{t->stream};  // the staging buffers stay with the trainer
    const int64_t *d_mindptr = nullptr;
    const int32_t *d_mindices = nullptr;
    // the fused tensor-core kernel walks each mask row with a cursor: column ids must ascend
    bool mask_sorted = true;
    if (mask_mode == 0) {
      if (t->X.sorted_state < 0)
        t->X.sorted_state =
            csr_rows_strictly_sorted(t->X.indptr.get(), t->X.indices.get(), t->X.n_rows, t->stream) ? 1 : 0;
      mask_sorted = t->X.sorted_state == 1;
    }
    if (mask_mode == 2) {
      stage_mask(rows, t->I, mask_indptr, mask_indices, t->rec_mindptr, t->rec_mindices, t->stream);
      for (int64_t r = 0; r < rows && mask_sorted; r++)
        for (int64_t j = mask_indptr[r] + 1; j < mask_indptr[r + 1]; j++)
          if (mask_indices[j - 1] >= mask_indices[j]) {
            mask_sorted = false;
            break;
          }
      d_mindptr = t->rec_mindptr.get();
      d_mindices = t->rec_mindices.get();
    }
    int32_t *d_idx = t->rec_idx.ensure(rows * k);
    float *d_sc = t->rec_score.ensure(rows * k);
    int32_t *d_cnt = t->rec_count.ensure(rows);
    // allow-lists (recommendable items): strictly ascending int32 lists, one shared or one per row
    int64_t *d_aindptr = nullptr;
    int32_t *d_aindices = nullptr;
    uint32_t *d_abitmap = nullptr;
    if (allow_n_lists > 0) {
      require(allow_n_lists == 1 || allow_n_lists == rows, "allow-lists: one shared list or one per row");
      require(allow_indptr != nullptr && allow_indptr[0] == 0, "allow indptr must start at 0");
      const int64_t annz = allow_indptr[allow_n_lists];
      require(annz == 0 || allow_indices != nullptr, "allow indices are null");
      for (int64_t r = 0; r < allow_n_lists; r++)
        for (int64_t j = allow_indptr[r]; j < allow_indptr[r + 1]; j++) {
          require(allow_indices[j] >= 0 && allow_indices[j] < t->I, "allowed item out of range");
          require(j == allow_indptr[r] || allow_indices[j - 1] < allow_indices[j],
                  "allow-lists must be strictly ascending");
        }
      if (allow_n_lists == 1) {  // a shared list goes to the kernel as a bitmap of the catalogue
        std::vector<uint32_t> &words = t->rec_abitmap_host;  // outlives the asynchronous copy
        words.assign((size_t)((t->I + 31) / 32), 0u);
        for (int64_t j = 0; j < annz; j++) words[allow_indices[j] >> 5] |= 1u << (allow_indices[j] & 31);
        d_abitmap = reinterpret_cast<uint32_t *>(t->rec_aindices.ensure(words.size()));
        CUDA_CHECK(cudaMemcpyAsync(d_abitmap, words.data(), sizeof(uint32_t) * words.size(),
                                   cudaMemcpyHostToDevice, t->stream));
      } else {
        d_aindptr = t->rec_aindptr.ensure(allow_n_lists + 1);
        d_aindices = t->rec_aindices.ensure(std::max<int64_t>(annz, 1));
        CUDA_CHECK(cudaMemcpyAsync(d_aindptr, allow_indptr, sizeof(int64_t) * (allow_n_lists + 1),
                                   cudaMemcpyHostToDevice, t->stream));
        if (annz)
          CUDA_CHECK(cudaMemcpyAsync(d_aindices, allow_indices, sizeof(int32_t) * annz, cudaMemcpyHostToDevice,
                                     t->stream));
      }
    }
    const bool fused = score_tc_supported(t->ld, k) && mask_sorted;
    // users picked by index: their factor rows are gathered into a dense block first
    const float *user_rows = t->factor[0].get() + begin * t->ld;
    int64_t *d_uidx = nullptr;
    if (user_idx != nullptr) {
      d_uidx = t->rec_uidx.ensure(rows);
      float *gathered = t->rec_users.ensure(rows * t->ld);
      CUDA_CHECK(cudaMemcpyAsync(d_uidx, user_idx, sizeof(int64_t) * rows, cudaMemcpyHostToDevice, t->stream));
      launch_gather_rows(t->factor[0].get(), t->ld, d_uidx, rows, gathered, t->stream);
      user_rows = gathered;
      if (mask_mode == 0 && !fused)
        throw NotImplemented("mask='train' for users picked by index needs the fused tensor-core kernel");
    }
    if (user_emb != nullptr) {  // host embeddings [rows x K] -> padded device rows [rows x ld]
      float *staged = t->rec_emb.ensure(rows * t->K);
      float *padded = t->rec_users.ensure(rows * t->ld);
      CUDA_CHECK(cudaMemcpyAsync(staged, user_emb, sizeof(float) * rows * t->K, cudaMemcpyHostToDevice, t->stream));
      launch_pad_copy(staged, rows, (int)t->K, padded, t->ld, t->stream);
      user_rows = padded;
    }
    if (allow_n_lists > 0 && !fused)
      throw NotImplemented("allow-lists need the fused tensor-core kernel (row stride <= 128, cutoff <= 128, "
                           "sorted mask rows)");
    if (fused) {
      // scores + mask + top-k in one tcgen05 kernel; only candidate keys touch HBM
      const int64_t slab_rows = std::max<int64_t>(128, ((1ll << 29) / (8 * 256)) / 128 * 128);
      for (int64_t b = 0; b < rows; b += slab_rows) {
        const int64_t m = std::min(slab_rows, rows - b);
        void *scratch = ensure_score_buf(t, score_tc_scratch_bytes(m, t->I, k));
        const int64_t *mip = nullptr;
        const int32_t *mix = nullptr;
        const float *mdt = nullptr;
        int64_t mrow0 = 0;
        const int64_t *mrowmap = nullptr;
        if (mask_mode == 0) {
          mip = t->X.indptr.get(); mix = t->X.indices.get(); mdt = t->X.data.get();
          mrow0 = begin + b - t->X.row_base;
          if (d_uidx) { mrowmap = d_uidx + b; mrow0 = -t->X.row_base; }
        } else if (mask_mode == 2) {
          mip = d_mindptr; mix = d_mindices; mrow0 = b;
        }
        launch_score_topk_tc(user_rows + b * t->ld, m, t->factor[1].get(), t->I, t->ld, mip,
                             mix, mdt, mrow0, (int)k, scratch, d_idx + b * k, d_sc + b * k,
                             d_cnt + b, t->stream, (int)std::min<int64_t>(allow_n_lists, 2), d_aindptr,
                             d_aindices, b, d_abitmap, mrowmap);
      }
    }
    const int64_t slab = std::max<int64_t>(1, std::min<int64_t>(rows, (1ll << 29) / (4 * t->I)));
    float *buf = fused ? nullptr : ensure_score_buf(t, sizeof(float) * slab * t->I);
    for (int64_t b = 0; b < rows && !fused; b += slab) {
      const int64_t m = std::min(slab, rows - b);
      launch_scores(user_rows + b * t->ld, m, t->factor[1].get(), t->I, t->ld, buf, t->I, t->stream);
      if (mask_mode == 0)
        launch_mask_rows(buf, t->I, t->X.indptr.get(), t->X.indices.get(), t->X.data.get(),
                         begin + b - t->X.row_base, m, 0, t->stream);
      else if (mask_mode == 2)
        launch_mask_rows(buf, t->I, d_mindptr, d_mindices, nullptr, b, m, 0, t->stream);
      launch_topk_rows(buf, t->I, m, t->I, (int)k, d_idx + b * k, d_sc + b * k, d_cnt + b,
                       t->stream);
    }
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
    // one allocation: rec | count | gt indptr | gt indices | discount | cum | acc[5] | valid | item_cnt
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; };
    const size_t o_rec = take(sizeof(int32_t) * rows * k), o_cnt = take(sizeof(int32_t) * rows),
                 o_ip = take(sizeof(int64_t) * (rows + 1)), o_ix = take(sizeof(int32_t) * std::max<int64_t>(gnnz, 1)),
                 o_d = take(sizeof(double) * k), o_c = take(sizeof(double) * k), o_acc = take(sizeof(double) * 5),
                 o_v = take(sizeof(unsigned long long)), o_ic = take(sizeof(unsigned long long) * n_items);
    DeviceBuffer<char> buf;
    StreamSyncOnExit sync{s};
    char *d = buf.alloc(off);
    CUDA_CHECK(cudaMemcpyAsync(d + o_rec, rec, sizeof(int32_t) * rows * k, cudaMemcpyHostToDevice, s));
    CUDA_CHECK(cudaMemcpyAsync(d + o_cnt, count, sizeof(int32_t) * rows, cudaMemcpyHostToDevice, s));
    CUDA_CHECK(cudaMemcpyAsync(d + o_ip, gt_indptr, sizeof(int64_t) * (rows + 1), cudaMemcpyHostToDevice, s));
    if (gnnz) CUDA_CHECK(cudaMemcpyAsync(d + o_ix, gt_indices, sizeof(int32_t) * gnnz, cudaMemcpyHostToDevice, s));
    CUDA_CHECK(cudaMemcpyAsync(d + o_d, discount, sizeof(double) * k, cudaMemcpyHostToDevice, s));
    CUDA_CHECK(cudaMemcpyAsync(d + o_c, cum.data(), sizeof(double) * k, cudaMemcpyHostToDevice, s));
    CUDA_CHECK(cudaMemsetAsync(d + o_acc, 0, off - o_acc, s));
    launch_metrics_rows(reinterpret_cast<int32_t *>(d + o_rec), reinterpret_cast<int32_t *>(d + o_cnt), rows, (int)k,
                        reinterpret_cast<int64_t *>(d + o_ip), reinterpret_cast<int32_t *>(d + o_ix),
                        reinterpret_cast<double *>(d + o_d), reinterpret_cast<double *>(d + o_c),
                        recall_with_cutoff, reinterpret_cast<double *>(d + o_acc),
                        reinterpret_cast<unsigned long long *>(d + o_v),
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
