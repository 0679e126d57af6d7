// Ranking metrics of recommendation lists on the device: the bookkeeping of
// EvaluatorCore::get_metrics_local + Metrics::update (/root/reference/cpp_source/evaluator.cpp:127-166,
// 308-361) for lists that the fused top-k kernel (score_tc.cu) or the SIMT top-k (score.cu) has
// already produced, and the diversity part of Metrics::as_dict (:87-123) on a histogram.
// The reference walks the users on host threads; a numpy restatement of that loop (np.isin over
// rows * cutoff keys) took ~3 s for the 138 493 users of configs[1] next to 8 ms of scoring.
//
// One warp per user, several cutoffs in one pass: a list of length max(cutoffs) serves every
// shorter cutoff as its prefix.  Lane j takes position j of the list (32 positions per step):
//   hit_j = rec_j in the user's ground-truth row (binary search; the row is sorted),
//   dcg_j = hit_j * discount_j,   ap_j = hit_j * (hits up to j) / (j + 1),
// and an inclusive warp scan turns them into prefix sums over the list.  Lane c (< n_cut) owns cutoff
// c: it picks the prefix at n_rec_c - 1, n_rec_c = min(count, cutoffs[c]), and accumulates
//   hit += (hits > 0), precision += hits / n_rec, recall += hits / n_gt (or min(n_gt, n_rec)),
//   ndcg += dcg / idcg(min(n_gt, n_rec)), map += ap / n_gt
// -- users without ground truth are skipped (:319-321), users without recommendable items only
// count as valid (:131-133).  item_cnt[c][rec_j] += 1 for every cutoff that covers position j.
// All sums are float64 (the reference's); discount_j = 1 / log2(2 + j) and its prefix sums come from
// the host so that both sides use the very same table.
//
// Determinism: early stopping compares these sums between passes, so no float64 atomics.  Each CTA
// adds its warps' sums in warp order into its own partial; metrics_reduce_kernel adds the partials in
// CTA order.  The grid is a function of the row count only, so the same chunks give the same bits.
// The histograms and valid_user are integers (atomics are exact).
#include "common.cuh"

namespace ials {
namespace {

constexpr int kMetricsThreads = 256;
constexpr int kMetricsWarps = kMetricsThreads / kWarp;
constexpr int kMaxGridMetrics = kNumSMsB200 * 16;

__global__ void __launch_bounds__(kMetricsThreads)
metrics_rows_kernel(const int32_t *__restrict__ rec, const int32_t *__restrict__ cnt, int64_t rows, int k,
                    const int64_t *__restrict__ gt_indptr, const int32_t *__restrict__ gt_indices,
                    const double *__restrict__ discount, const double *__restrict__ cum_discount,
                    const int32_t *__restrict__ cutoffs, int n_cut, int recall_with_cutoff, int64_t n_items,
                    double *__restrict__ partial /*[grid][n_cut][5]*/, unsigned long long *valid_user /*[n_cut]*/,
                    unsigned long long *item_cnt /*[n_cut][n_items]*/) {
  __shared__ double s_acc[kMetricsWarps][kWarp][5];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int my_cut = lane < n_cut ? cutoffs[lane] : 0;
  double a_hit = 0, a_recall = 0, a_ndcg = 0, a_map = 0, a_prec = 0;
  unsigned long long a_valid = 0;
  for (int64_t u = warp; u < rows; u += n_warps) {
    const int64_t g0 = gt_indptr[u], g1 = gt_indptr[u + 1];
    const int64_t n_gt = g1 - g0;
    if (n_gt == 0) continue;
    a_valid++;
    const int n_rec = min(cnt[u], k);
    if (n_rec <= 0) continue;
    const int my_n = min(n_rec, my_cut);  // 0 on lanes without a cutoff
    double run_dcg = 0, run_ap = 0, my_dcg = 0, my_ap = 0;
    int run_hits = 0, my_hits = 0;
    for (int base = 0; base < n_rec; base += 32) {
      const int j = base + lane;
      const int item = j < n_rec ? rec[u * k + j] : -1;
      bool hit = false;
      if (item >= 0) {
        int64_t lo = g0, hi = g1;
        while (lo < hi) {
          const int64_t mid = (lo + hi) >> 1;
          if (gt_indices[mid] < item) lo = mid + 1; else hi = mid;
        }
        hit = lo < g1 && gt_indices[lo] == item;
        for (int c = 0; c < n_cut; c++)
          if (j < cutoffs[c]) atomicAdd(&item_cnt[c * n_items + item], 1ull);
      }
      const unsigned ballot = __ballot_sync(0xffffffffu, hit);
      const int upto = run_hits + __popc(ballot & (0xffffffffu >> (31 - lane)));
      double d = hit ? discount[j] : 0.0, a = hit ? (double)upto / (double)(j + 1) : 0.0;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {  // inclusive scan over the 32 positions
        const double dn = __shfl_up_sync(0xffffffffu, d, o), an = __shfl_up_sync(0xffffffffu, a, o);
        if (lane >= o) { d += dn; a += an; }
      }
      d += run_dcg;
      a += run_ap;
      // the lanes whose cutoff ends inside this step take the prefix at their last position
      const int src = my_n - 1 - base;
      const bool ends_here = src >= 0 && src < 32;
      const double pd = __shfl_sync(0xffffffffu, d, src & 31), pa = __shfl_sync(0xffffffffu, a, src & 31);
      if (ends_here) {
        my_dcg = pd;
        my_ap = pa;
        my_hits = run_hits + __popc(ballot & (0xffffffffu >> (31 - src)));
      }
      run_dcg = __shfl_sync(0xffffffffu, d, 31);
      run_ap = __shfl_sync(0xffffffffu, a, 31);
      run_hits += __popc(ballot);
    }
    if (my_n > 0) {
      const int64_t lim = min(n_gt, (int64_t)my_n);
      a_hit += my_hits > 0 ? 1.0 : 0.0;
      a_prec += (double)my_hits / (double)my_n;
      a_recall += (double)my_hits / (double)(recall_with_cutoff ? lim : n_gt);
      a_ndcg += my_dcg / cum_discount[lim - 1];
      a_map += my_ap / (double)n_gt;
    }
  }
  if (lane < n_cut && a_valid) atomicAdd(&valid_user[lane], a_valid);
  s_acc[wib][lane][0] = a_hit;
  s_acc[wib][lane][1] = a_recall;
  s_acc[wib][lane][2] = a_ndcg;
  s_acc[wib][lane][3] = a_map;
  s_acc[wib][lane][4] = a_prec;
  __syncthreads();
  if (threadIdx.x < n_cut * 5) {  // (cutoff, metric) pairs: the warps' sums in warp order
    const int c = threadIdx.x / 5, m = threadIdx.x % 5;
    double s = 0;
    for (int w = 0; w < kMetricsWarps; w++) s += s_acc[w][c][m];
    partial[(int64_t)blockIdx.x * n_cut * 5 + threadIdx.x] = s;
  }
}

// acc[c][m] += sum over CTAs (in CTA order) of partial[cta][c][m]; total_user[c] += rows
__global__ void metrics_reduce_kernel(const double *__restrict__ partial, int n_parts, int n_cut, int64_t rows,
                                      double *acc, unsigned long long *total_user) {
  const int t = threadIdx.x;
  if (t < n_cut * 5) {
    double s = 0;
    for (int p = 0; p < n_parts; p++) s += partial[(int64_t)p * n_cut * 5 + t];
    acc[t] += s;
  }
  if (t < n_cut) total_user[t] += (unsigned long long)rows;
}

// ---- diversity of a histogram (Metrics::as_dict without the sort) ----
// Sorted ascending, the items of count v occupy the ranks [R_v, R_v + m_v), m_v = #items of count v,
// R_v = #items of count < v.  So  sum_r (2 r - n + 1) cnt_r = sum_v v m_v (2 R_v + m_v - n), exactly in
// 128-bit integers, and  entropy = sum_v m_v (-log(v / T) v / T).

constexpr int kDivThreads = 256;
constexpr int kDivBlocks = kNumSMsB200 * 2;

// stats = {total, appeared, max}
__global__ void hist_stats_kernel(const unsigned long long *__restrict__ h, int64_t n, unsigned long long *stats) {
  unsigned long long tot = 0, app = 0, mx = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const unsigned long long v = h[i];
    tot += v;
    app += v > 0;
    mx = v > mx ? v : mx;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    tot += __shfl_xor_sync(0xffffffffu, tot, o);
    app += __shfl_xor_sync(0xffffffffu, app, o);
    const unsigned long long m2 = __shfl_xor_sync(0xffffffffu, mx, o);
    mx = m2 > mx ? m2 : mx;
  }
  if ((threadIdx.x & 31) == 0 && tot) {
    atomicAdd(&stats[0], tot);
    atomicAdd(&stats[1], app);
    atomicMax(&stats[2], mx);
  }
}

// table[v] = number of items with count v (v >= 1)
__global__ void count_of_counts_kernel(const unsigned long long *__restrict__ h, int64_t n,
                                       unsigned long long *table) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    if (h[i]) atomicAdd(&table[h[i]], 1ull);
}

__device__ __forceinline__ int64_t seg_begin(int64_t len, int parts, int p) { return len * p / parts; }

// bsum[b] = sum of table over block b's segment
__global__ void __launch_bounds__(kDivThreads)
table_block_sums_kernel(const unsigned long long *__restrict__ table, int64_t len, unsigned long long *bsum) {
  __shared__ unsigned long long s[kDivThreads / kWarp];
  const int64_t b0 = seg_begin(len, gridDim.x, blockIdx.x), b1 = seg_begin(len, gridDim.x, blockIdx.x + 1);
  unsigned long long v = 0;
  for (int64_t i = b0 + threadIdx.x; i < b1; i += blockDim.x) v += table[i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long t = 0;
    for (int w = 0; w < kDivThreads / kWarp; w++) t += s[w];
    bsum[blockIdx.x] = t;
  }
}

// Each block walks its segment of the table in rank order: thread t takes a contiguous sub-segment,
// a block scan of the sub-segment counts gives every entry its R_v.  Per block: the exact Gini sum
// and the entropy (sub-segments added in thread order) -> part_gini[b], part_ent[b].
__global__ void __launch_bounds__(kDivThreads)
table_terms_kernel(const unsigned long long *__restrict__ table, int64_t len, const unsigned long long *__restrict__ bsum,
                   const unsigned long long *__restrict__ stats, int64_t n_items, __int128 *part_gini,
                   double *part_ent) {
  __shared__ unsigned long long s_cnt[kDivThreads];
  __shared__ __int128 s_gini[kDivThreads];
  __shared__ double s_ent[kDivThreads];
  const int64_t b0 = seg_begin(len, gridDim.x, blockIdx.x), b1 = seg_begin(len, gridDim.x, blockIdx.x + 1);
  const int64_t t0 = b0 + (b1 - b0) * threadIdx.x / blockDim.x, t1 = b0 + (b1 - b0) * (threadIdx.x + 1) / blockDim.x;
  unsigned long long mine = 0;
  for (int64_t v = t0; v < t1; v++) mine += table[v];
  s_cnt[threadIdx.x] = mine;
  __syncthreads();
  unsigned long long R = (unsigned long long)n_items - stats[1];  // the items of count 0 come first
  for (int b = 0; b < (int)blockIdx.x; b++) R += bsum[b];
  for (int t = 0; t < (int)threadIdx.x; t++) R += s_cnt[t];
  const double total = (double)stats[0];
  __int128 gini = 0;
  double ent = 0;
  for (int64_t v = t0; v < t1; v++) {
    const unsigned long long m = table[v];
    if (!m) continue;
    gini += (__int128)v * (__int128)m * ((__int128)2 * R + (__int128)m - (__int128)n_items);
    const double p = (double)v / total;
    ent += (double)m * (-log(p) * p);
    R += m;
  }
  s_gini[threadIdx.x] = gini;
  s_ent[threadIdx.x] = ent;
  __syncthreads();
  if (threadIdx.x == 0) {
    __int128 g = 0;
    double e = 0;
    for (int t = 0; t < (int)blockDim.x; t++) { g += s_gini[t]; e += s_ent[t]; }
    part_gini[blockIdx.x] = g;
    part_ent[blockIdx.x] = e;
  }
}

// out = {appeared_item, entropy, gini_index}
__global__ void diversity_finish_kernel(const __int128 *__restrict__ part_gini, const double *__restrict__ part_ent,
                                        int n_parts, const unsigned long long *__restrict__ stats, int64_t n_items,
                                        double *out) {
  __int128 g = 0;
  double e = 0;
  for (int p = 0; p < n_parts; p++) { g += part_gini[p]; e += part_ent[p]; }
  double gini = (double)g;
  if (stats[0] > 0) gini /= (double)n_items * (double)stats[0];
  out[0] = (double)stats[1];
  out[1] = e;
  out[2] = gini;
}

}  // namespace

int64_t metrics_partials(int64_t rows) {
  return std::max<int64_t>(1, std::min<int64_t>(ceil_div(rows * kWarp, kMetricsThreads), kMaxGridMetrics));
}

void launch_metrics_rows(const int32_t *rec, const int32_t *cnt, int64_t rows, int k, const int64_t *gt_indptr,
                         const int32_t *gt_indices, const double *discount, const double *cum_discount,
                         const int32_t *cutoffs, int n_cut, int recall_with_cutoff, int64_t n_items,
                         double *partial, double *acc, unsigned long long *valid_user,
                         unsigned long long *total_user, unsigned long long *item_cnt, cudaStream_t s) {
  if (rows == 0) return;
  if (n_cut < 1 || n_cut > kMaxMetricsCutoffs) throw InvalidArgument("metrics: 1 .. 32 cutoffs per launch");
  const unsigned grid = (unsigned)metrics_partials(rows);
  metrics_rows_kernel<<<grid, kMetricsThreads, 0, s>>>(rec, cnt, rows, k, gt_indptr, gt_indices, discount,
                                                       cum_discount, cutoffs, n_cut, recall_with_cutoff, n_items,
                                                       partial, valid_user, item_cnt);
  count_launch();
  CUDA_CHECK(cudaGetLastError());
  metrics_reduce_kernel<<<1, kMaxMetricsCutoffs * 5, 0, s>>>(partial, (int)grid, n_cut, rows, acc, total_user);
  count_launch();
  CUDA_CHECK(cudaGetLastError());
}

void diversity_of_histogram(const unsigned long long *hist, int64_t n_items, DeviceBuffer<unsigned char> &ws,
                            double *d_out, cudaStream_t s) {
  // workspace: stats[3] | bsum[kDivBlocks] | part_gini[kDivBlocks] | part_ent[kDivBlocks] | table
  const size_t o_stats = 0, o_bsum = 64, o_pg = o_bsum + 8 * kDivBlocks, o_pe = o_pg + 16 * kDivBlocks,
               o_tab = round_up(o_pe + 8 * kDivBlocks, 256);
  unsigned char *w = ws.ensure(o_tab);
  auto *stats = reinterpret_cast<unsigned long long *>(w + o_stats);
  CUDA_CHECK(cudaMemsetAsync(stats, 0, 3 * sizeof(unsigned long long), s));
  const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>(ceil_div(n_items, 256), kNumSMsB200 * 8));
  if (n_items) {
    hist_stats_kernel<<<grid, 256, 0, s>>>(hist, n_items, stats);
    count_launch();
    CUDA_CHECK(cudaGetLastError());
  }
  unsigned long long h_stats[3];
  CUDA_CHECK(cudaMemcpyAsync(h_stats, stats, sizeof(h_stats), cudaMemcpyDeviceToHost, s));
  CUDA_CHECK(cudaStreamSynchronize(s));  // the table is as long as the largest count
  const int64_t len = (int64_t)h_stats[2] + 1;
  w = ws.ensure(o_tab + sizeof(unsigned long long) * len);  // may move: the stats are re-read below
  stats = reinterpret_cast<unsigned long long *>(w + o_stats);
  CUDA_CHECK(cudaMemcpyAsync(stats, h_stats, sizeof(h_stats), cudaMemcpyHostToDevice, s));
  auto *bsum = reinterpret_cast<unsigned long long *>(w + o_bsum);
  auto *pg = reinterpret_cast<__int128 *>(w + o_pg);
  auto *pe = reinterpret_cast<double *>(w + o_pe);
  auto *table = reinterpret_cast<unsigned long long *>(w + o_tab);
  CUDA_CHECK(cudaMemsetAsync(table, 0, sizeof(unsigned long long) * len, s));
  if (n_items) {
    count_of_counts_kernel<<<grid, 256, 0, s>>>(hist, n_items, table);
    count_launch();
  }
  table_block_sums_kernel<<<kDivBlocks, kDivThreads, 0, s>>>(table, len, bsum);
  table_terms_kernel<<<kDivBlocks, kDivThreads, 0, s>>>(table, len, bsum, stats, n_items, pg, pe);
  diversity_finish_kernel<<<1, 1, 0, s>>>(pg, pe, kDivBlocks, stats, n_items, d_out);
  count_launch(3);
  CUDA_CHECK(cudaGetLastError());
}

}  // namespace ials
