// Explanations behind the C ABI (ials_trainer_explain): each iALS score split into the contributions of
// the query row's history entries, solved on the device by the EXPLAIN instantiation of cholesky_tile.cu
// and selected per (row, target) pair by launch_topk_segments.
#include <algorithm>
#include <vector>

#include "trainer.cuh"

using namespace ials;

namespace {

// A call runs in slabs of at most this many scheduled rows, (row, target) pairs and contributions (pairs x
// history length; one row alone may hold more): they bound the pair outputs and the contribution scratch,
// 8 bytes per contribution with its column id.
constexpr int64_t kExplainSlabRows = 262144;
constexpr int64_t kExplainSlabPairs = 1ll << 22;
constexpr int64_t kExplainSlabContrib = 1ll << 25;

struct ExplainSlab {
  int64_t slot0 = 0, n_slots = 0, pair0 = 0, n_pairs = 0, n_contrib = 0, max_len = 0;
};

// A host CSR of `rows` rows over [0, n_cols): indptr from 0, non-decreasing, ids in range
void check_csr(int64_t rows, int64_t n_cols, const int64_t *indptr, const int32_t *indices, const char *what) {
  const std::string w(what);
  require(indptr != nullptr && indptr[0] == 0, (w + " indptr must start at 0").c_str());
  for (int64_t r = 0; r < rows; r++) require(indptr[r + 1] >= indptr[r], (w + " indptr must be non-decreasing").c_str());
  require(indptr[rows] == 0 || indices != nullptr, (w + " indices are null").c_str());
  for (int64_t j = 0; j < indptr[rows]; j++)
    require(indices[j] >= 0 && indices[j] < n_cols, (w + " index out of range").c_str());
}

template <typename T>
T *upload(DeviceBuffer<T> &d, const T *src, int64_t n, cudaStream_t s) {
  T *p = d.ensure(std::max<int64_t>(n, 1));
  if (n) CUDA_CHECK(cudaMemcpyAsync(p, src, sizeof(T) * n, cudaMemcpyHostToDevice, s));
  return p;
}

}  // namespace

extern "C" {

int ials_trainer_explain(ials_trainer *t, int side, const int64_t *query_idx, int64_t begin, int64_t end,
                         const int64_t *hist_indptr, const int32_t *hist_indices, const float *hist_data,
                         const int64_t *target_indptr, const int32_t *target_indices, int64_t n_top,
                         float *out_score, float *out_prior, int32_t *out_idx, float *out_contrib,
                         int32_t *out_count) {
  return guarded([&] {
    require(t != nullptr, "trainer is null");
    require_side(side);
    const bool cold = hist_indptr != nullptr;
    require(!(cold && query_idx != nullptr), "give rows by index or cold rows, not both");
    const int64_t n = t->n_rows(side), n_other = t->n_rows(1 - side);
    require(end >= begin && begin >= 0 && (query_idx != nullptr || cold ? begin == 0 : end <= n), "bad query block");
    require(n_top >= 1 && n_top <= 1024, "n_top must be in [1, 1024]");
    const int64_t rows = end - begin;
    check_csr(rows, n_other, target_indptr, target_indices, "target");
    if (cold) {
      check_csr(rows, n_other, hist_indptr, hist_indices, "history");
      require(hist_indptr[rows] == 0 || hist_data != nullptr, "history data are null");
    }
    const DeviceCsr &csr = side == 0 ? t->X : t->Xt;
    if (!cold && rows > 0) {
      if (!t->has_X) throw std::runtime_error("this trainer was restored without its interaction matrix: explain cold rows");
      for (int64_t r = 0; r < rows; r++) {
        const int64_t q = query_idx != nullptr ? query_idx[r] : begin + r;
        require(q >= 0 && q < n, "query index out of range");
        require(q >= csr.row_base && q < csr.row_base + csr.n_rows,
                "a row-sharded trainer explains only its own rows by index");
      }
    }
    ials_solver_config sc{};
    SolveArgs a = make_args(t, side, t->factor[side].get(), csr, &sc);
    if (!cholesky_tile_supported(a)) throw NotImplemented("explanations: n_components > 256 not supported");
    const int64_t n_pairs = target_indptr[rows];
    if (n_pairs == 0) return;
    require(out_score != nullptr && out_idx != nullptr && out_count != nullptr, "output pointer is null");
    DeviceGuard g(t->device);
    StreamSyncOnExit sync{t->stream};  // the staging buffers stay with the trainer

    // the history length of every query row (rows by index: from a host copy of the CSR's indptr)
    std::vector<int64_t> &ip = t->indptr_host[side];
    if (!cold && ip.empty()) {
      ip.resize((size_t)csr.n_rows + 1);
      CUDA_CHECK(cudaMemcpyAsync(ip.data(), csr.indptr.get(), sizeof(int64_t) * ip.size(), cudaMemcpyDeviceToHost,
                                 t->stream));
      CUDA_CHECK(cudaStreamSynchronize(t->stream));
    }
    // the schedule: rows with at least one target (CSR row of each slot), cut into slabs
    std::vector<int32_t> sched;
    std::vector<int64_t> len_of_slot, pairs_of_slot;
    std::vector<ExplainSlab> slabs;
    for (int64_t r = 0; r < rows; r++) {
      const int64_t nt = target_indptr[r + 1] - target_indptr[r];
      if (nt == 0) continue;
      const int64_t u = cold ? r : (query_idx != nullptr ? query_idx[r] : begin + r) - csr.row_base;
      const int64_t len = cold ? hist_indptr[r + 1] - hist_indptr[r] : ip[u + 1] - ip[u];
      if (slabs.empty() || slabs.back().n_slots == kExplainSlabRows || slabs.back().n_pairs + nt > kExplainSlabPairs ||
          slabs.back().n_contrib + nt * len > kExplainSlabContrib) {
        ExplainSlab c;
        c.slot0 = (int64_t)sched.size();
        c.pair0 = target_indptr[r];
        slabs.push_back(c);
      }
      ExplainSlab &c = slabs.back();
      c.n_slots++;
      c.n_pairs += nt;
      c.n_contrib += nt * len;
      c.max_len = std::max(c.max_len, len);
      sched.push_back((int32_t)u);
      len_of_slot.push_back(len);
      pairs_of_slot.push_back(nt);
    }
    // slab-local offsets: slot -> first pair (n_slots + 1), pair -> first contribution (n_pairs + 1); slab
    // i's runs start at slot0 + i and at n_sched + n_slabs + pair0 + i
    const int64_t n_sched = (int64_t)sched.size(), n_slabs = (int64_t)slabs.size();
    const int64_t cp0 = n_sched + n_slabs;
    std::vector<int64_t> offsets((size_t)(cp0 + n_pairs + n_slabs));
    int64_t max_pairs = 1, max_contrib = 1;
    for (int64_t i = 0; i < n_slabs; i++) {
      const ExplainSlab &c = slabs[i];
      int64_t *pp = offsets.data() + c.slot0 + i;
      int64_t *cp = offsets.data() + cp0 + c.pair0 + i;
      int64_t pair = 0, contrib = 0;
      for (int64_t k = 0; k < c.n_slots; k++) {
        pp[k] = pair;
        for (int64_t q = 0; q < pairs_of_slot[c.slot0 + k]; q++, contrib += len_of_slot[c.slot0 + k]) cp[pair++] = contrib;
      }
      pp[c.n_slots] = pair;
      cp[pair] = contrib;
      max_pairs = std::max(max_pairs, c.n_pairs);
      max_contrib = std::max(max_contrib, c.n_contrib);
    }
    const int32_t *d_sched = upload(t->expl_rows, sched.data(), n_sched, t->stream);
    const int64_t *d_off = upload(t->expl_offsets, offsets.data(), (int64_t)offsets.size(), t->stream);
    const int32_t *d_targets = upload(t->expl_targets, target_indices, n_pairs, t->stream);
    if (cold) {
      a.indptr = upload(t->expl_hist_indptr, hist_indptr, rows + 1, t->stream);
      a.indices = upload(t->expl_hist_indices, hist_indices, hist_indptr[rows], t->stream);
      a.data = upload(t->expl_hist_data, hist_data, hist_indptr[rows], t->stream);
      a.n_rows = rows;
      a.row_base = 0;
    } else if (side_uses_features(t, side)) {  // the stored prior of the rank's own rows, as a step uses it
      check_feature_weight_shapes(t, false);
      a.prior = stored_prior(t, side) - csr.row_base * t->ld;
    }
    float *d_pair = t->expl_pair_out.ensure(2 * max_pairs);  // score | prior
    float *d_contrib = t->expl_contrib.ensure(max_contrib);
    int32_t *d_cidx = t->expl_contrib_idx.ensure(max_contrib);
    int32_t *d_idx = t->rec_idx.ensure(max_pairs * n_top);
    float *d_sc = t->rec_score.ensure(max_pairs * n_top);
    int32_t *d_cnt = t->rec_count.ensure(max_pairs);
    gram_side(t, side);  // P from the other side as it is now
    for (int64_t i = 0; i < n_slabs; i++) {
      const ExplainSlab &c = slabs[i];
      SolveArgs sa = a;
      sa.order = d_sched + c.slot0;
      sa.n_sched = c.n_slots;
      SubspaceArgs ex{};
      ex.pair_ptr = d_off + c.slot0 + i;
      ex.targets = d_targets + c.pair0;
      ex.contrib_ptr = d_off + cp0 + c.pair0 + i;
      ex.score = d_pair;
      ex.prior = out_prior != nullptr ? d_pair + max_pairs : nullptr;
      ex.contrib = d_contrib;
      ex.contrib_idx = d_cidx;
      launch_explain_tile(sa, ex, t->stream);
      launch_topk_segments(d_contrib, CandSegments{ex.contrib_ptr, d_cidx, 0, 0, -1}, c.n_pairs, c.max_len,
                           (int)n_top, d_idx, d_sc, d_cnt, t->stream);
      auto down = [&](void *dst, const void *src, size_t bytes) {
        CUDA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, t->stream));
      };
      down(out_score + c.pair0, d_pair, sizeof(float) * c.n_pairs);
      if (out_prior) down(out_prior + c.pair0, ex.prior, sizeof(float) * c.n_pairs);
      down(out_idx + c.pair0 * n_top, d_idx, sizeof(int32_t) * c.n_pairs * n_top);
      if (out_contrib) down(out_contrib + c.pair0 * n_top, d_sc, sizeof(float) * c.n_pairs * n_top);
      down(out_count + c.pair0, d_cnt, sizeof(int32_t) * c.n_pairs);
    }
    sync_and_check(t);  // a failed factorisation raises as a Cholesky step does
  });
}

}  // extern "C"
