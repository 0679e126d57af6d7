// Ranking of caller-given candidates: the scores of each query row against its own list of items
// (gathered dot products, cand_scores_kernel) and the top-k of each list (topk_segments_kernel, the
// threshold filter of score.cu's dense top-k over a segment).  The cost follows the number of
// (row, candidate) pairs, not the catalogue.
#include <algorithm>

#include <cub/warp/warp_merge_sort.cuh>

#include "topk.cuh"

namespace ials {
namespace {

constexpr int kCandThreads = 256;
constexpr int kWarpTkItems = 8;
constexpr int kWarpTkMax = kWarp * kWarpTkItems;  // longest list the warp-per-row selection takes

// The NI = ld / 32 floats of a row held by one lane: float4 slices when ld is a multiple of 128,
// else one float per 32-column stripe.  Queries and items use the same layout.
template <int NI>
__device__ __forceinline__ void load_row(const float *__restrict__ row, int lane, float (&v)[NI]) {
  if constexpr (NI % 4 == 0) {
#pragma unroll
    for (int m = 0; m < NI / 4; m++) {
      const float4 f = __ldg(reinterpret_cast<const float4 *>(row + m * 128 + lane * 4));
      v[4 * m] = f.x; v[4 * m + 1] = f.y; v[4 * m + 2] = f.z; v[4 * m + 3] = f.w;
    }
  } else {
#pragma unroll
    for (int i = 0; i < NI; i++) v[i] = __ldg(row + lane + 32 * i);
  }
}

// Is `item` hidden by the mask row [s, e)?  A stored zero hides nothing.
__device__ __forceinline__ bool masked(const CandMask &m, int64_t s, int64_t e, int32_t item) {
  if (m.sorted) {
    int64_t lo = s, hi = e;
    while (lo < hi) {  // first position whose id is >= item
      const int64_t mid = (lo + hi) >> 1;
      if (m.indices[mid] < item) lo = mid + 1; else hi = mid;
    }
    return lo < e && m.indices[lo] == item && (m.data == nullptr || m.data[lo] != 0.f);
  }
  for (int64_t j = s; j < e; j++)
    if (m.indices[j] == item && (m.data == nullptr || m.data[j] != 0.f)) return true;
  return false;
}

// One warp per (row, chunk of kCandChunk candidates): task g of the slab is chunk g - tasks[r] of the row r
// with tasks[r] <= g < tasks[r + 1], so only chunks that hold candidates are visited.  The query row sits
// in registers; for each group of up to 32 candidates every lane forms its partial dot product with each
// candidate row (read coalesced), then a transpose-reduce leaves the full score of candidate `lane` in
// lane `lane`: 31 shuffles per 32 scores.
template <int NI>
__global__ void __launch_bounds__(kCandThreads)
cand_scores_kernel(const float *__restrict__ queries, int ld, const float *__restrict__ item, CandSegments seg,
                   CandMask mask, const int64_t *__restrict__ tasks, int64_t n_rows, int64_t n_tasks,
                   float *__restrict__ scores) {
  // candidate rows loaded ahead of their products (a divisor of 32; ptxas -v shows no spills with these)
  constexpr int kBatch = NI == 3 ? 2 : NI <= 4 ? 8 : NI == 8 ? 4 : NI == 6 ? 1 : 2;
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x % kWarp;
  const int64_t stride = (int64_t)gridDim.x * (kCandThreads / kWarp), t0 = tasks[0];
  for (int64_t task = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / kWarp; task < n_tasks; task += stride) {
    const int64_t g = t0 + task;
    int64_t r = 0, hi = n_rows;  // the last row whose first task is <= g
    while (hi - r > 1) {
      const int64_t mid = (r + hi) >> 1;
      if (tasks[mid] <= g) r = mid; else hi = mid;
    }
    const int64_t c0 = (g - tasks[r]) * kCandChunk;
    const int64_t b = seg.begin(r), n = seg.end(r) - b;
    float q[NI];
    load_row<NI>(queries + r * ld, lane, q);
    int64_t ms = 0, me = 0;
    if (mask.indptr != nullptr) {
      const int64_t mr = mask.rowmap != nullptr ? mask.rowmap[r] + mask.row0 : mask.row0 + r;
      ms = mask.indptr[mr];
      me = mask.indptr[mr + 1];
    }
    const int32_t *ids = seg.indices + b;
    float *out = scores + seg.out(r);
    const int64_t c1 = min(n, c0 + kCandChunk);
    for (int64_t c = c0; c < c1; c += kWarp) {
      const int m = (int)min((int64_t)kWarp, c1 - c);
      const int32_t mine = ids[c + (lane < m ? lane : 0)];  // lanes past the list repeat candidate 0
      float p[kWarp];
#pragma unroll
      for (int e = 0; e < kWarp; e++) p[e] = 0.f;
#pragma unroll
      for (int e0 = 0; e0 < kWarp; e0 += kBatch) {  // kBatch candidate rows in flight per warp
        if (e0 >= m) break;  // warp-uniform: a group shorter than 32 loads only its own rows
        float v[kBatch][NI];
#pragma unroll
        for (int g = 0; g < kBatch; g++) load_row<NI>(item + (int64_t)__shfl_sync(full, mine, e0 + g) * ld, lane, v[g]);
#pragma unroll
        for (int g = 0; g < kBatch; g++) {
          float s = 0.f;
#pragma unroll
          for (int i = 0; i < NI; i++) s = fmaf(q[i], v[g][i], s);
          p[e0 + g] = s;
        }
      }
      // after the step of width w, p[i] (i < w) is candidate i + (lane & (32 - w)), summed over the
      // lanes that differ from this one in the bits from log2(w) up
#pragma unroll
      for (int w = kWarp / 2; w >= 1; w /= 2) {
        const bool upper = (lane & w) != 0;
#pragma unroll
        for (int i = 0; i < w; i++) {
          const float send = upper ? p[i] : p[i + w];
          const float keep = upper ? p[i + w] : p[i];
          p[i] = keep + __shfl_xor_sync(full, send, w);
        }
      }
      if (lane < m) out[c + lane] = (mask.indptr != nullptr && masked(mask, ms, me, mine)) ? -INFINITY : p[0];
    }
  }
}

// Row r of a slab: its segment of the score scratch, the item ids of its list as the column ids
struct SegmentRows {
  CandSegments seg;
  const float *scores;
  struct Row {
    const float *s;
    const int32_t *ids;
    int64_t n;
    __device__ float score(int64_t j) const { return s[j]; }
    __device__ uint32_t id(int64_t j) const { return (uint32_t)ids[j]; }
  };
  __device__ Row row(int64_t r) const {
    const int64_t b = seg.begin(r);
    return {scores + seg.out(r), seg.indices + b, seg.end(r) - b};
  }
};

// Lists of at most kWarpTkMax candidates: one warp per row sorts the row's keys in registers (a warp
// merge sort of kWarpTkItems keys per lane) instead of a CTA and its 2048-key radix sort.  Same keys,
// order, padding and counts as topk_segments_kernel.
struct KeyLess {
  __device__ bool operator()(unsigned long long a, unsigned long long b) const { return a < b; }
};
__global__ void __launch_bounds__(kCandThreads)
topk_segments_warp_kernel(SegmentRows rows, int64_t n_rows, int k, int32_t *__restrict__ out_idx,
                          float *__restrict__ out_score, int32_t *__restrict__ out_count) {
  using Sort = cub::WarpMergeSort<unsigned long long, kWarpTkItems, kWarp>;
  __shared__ typename Sort::TempStorage tmp[kCandThreads / kWarp];
  const int lane = threadIdx.x % kWarp, warp = threadIdx.x / kWarp;
  const int64_t stride = (int64_t)gridDim.x * (kCandThreads / kWarp);
  for (int64_t row = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / kWarp; row < n_rows; row += stride) {
    const auto src = rows.row(row);
    unsigned long long keys[kWarpTkItems];
    int valid = 0;
#pragma unroll
    for (int i = 0; i < kWarpTkItems; i++) {
      const int64_t j = i * kWarp + lane;  // coalesced; the sort does not care where a key starts
      keys[i] = ~0ull;
      if (j < src.n) {
        const float sc = src.score(j);
        if (sc != -INFINITY) { keys[i] = make_key(sc, src.id(j)); valid++; }
      }
    }
    Sort(tmp[warp]).Sort(keys, KeyLess());
#pragma unroll
    for (int o = kWarp / 2; o >= 1; o /= 2) valid += __shfl_xor_sync(0xffffffffu, valid, o);
    const int n_out = min(valid, k);
#pragma unroll
    for (int i = 0; i < kWarpTkItems; i++) {  // blocked: lane l holds sorted positions l * kWarpTkItems + i
      const int pos = lane * kWarpTkItems + i;
      if (pos < k) {
        const bool ok = pos < n_out;
        out_idx[row * k + pos] = ok ? (int32_t)(keys[i] & 0xffffffffu) : -1;
        if (out_score) out_score[row * k + pos] = ok ? key_score(keys[i]) : -INFINITY;
      }
    }
    for (int pos = kWarpTkMax + lane; pos < k; pos += kWarp) {
      out_idx[row * k + pos] = -1;
      if (out_score) out_score[row * k + pos] = -INFINITY;
    }
    if (lane == 0) out_count[row] = n_out;
    __syncwarp();  // the next row's sort reuses tmp[warp]
  }
}

__global__ void __launch_bounds__(kTkThreads)
topk_segments_kernel(SegmentRows rows, int64_t n_rows, int k, int32_t *__restrict__ out_idx,
                     float *__restrict__ out_score, int32_t *__restrict__ out_count) {
  topk_rows_body(rows, n_rows, k, out_idx, out_score, out_count);
}

template <int NI>
void launch_cand_scores_ni(const float *queries, int64_t n_rows, int ld, const float *item, const CandSegments &seg,
                           const int64_t *tasks, int64_t n_tasks, const CandMask &mask, float *scores, cudaStream_t s) {
  const int64_t per_block = kCandThreads / kWarp;
  const unsigned grid = (unsigned)std::min<int64_t>(ceil_div(n_tasks, per_block), (int64_t)kNumSMsB200 * 16);
  cand_scores_kernel<NI><<<grid, kCandThreads, 0, s>>>(queries, ld, item, seg, mask, tasks, n_rows, n_tasks, scores);
  count_launch();
}

}  // namespace

void launch_cand_scores(const float *queries, int64_t n_rows, int ld, const float *item, const CandSegments &seg,
                        const int64_t *tasks, int64_t n_tasks, const CandMask &mask, float *scores, cudaStream_t s) {
  if (n_rows == 0 || n_tasks == 0) return;
  if (ld % kWarp != 0 || ld < kWarp || ld > 16 * kWarp) throw InvalidArgument("candidate scores: ld must be 32 .. 512");
  switch (ld / kWarp) {
#define IALS_CAND_NI(ni) \
  case ni: launch_cand_scores_ni<ni>(queries, n_rows, ld, item, seg, tasks, n_tasks, mask, scores, s); break;
    IALS_CAND_NI(1) IALS_CAND_NI(2) IALS_CAND_NI(3) IALS_CAND_NI(4) IALS_CAND_NI(5) IALS_CAND_NI(6)
    IALS_CAND_NI(7) IALS_CAND_NI(8) IALS_CAND_NI(9) IALS_CAND_NI(10) IALS_CAND_NI(11) IALS_CAND_NI(12)
    IALS_CAND_NI(13) IALS_CAND_NI(14) IALS_CAND_NI(15) IALS_CAND_NI(16)
#undef IALS_CAND_NI
  }
  CUDA_CHECK(cudaGetLastError());
}

void launch_topk_segments(const float *scores, const CandSegments &seg, int64_t n_rows, int64_t max_len, int k,
                          int32_t *out_idx, float *out_score, int32_t *out_count, cudaStream_t s) {
  if (n_rows == 0) return;
  if (k < 1 || k > kTkCap - kTkChunk) throw InvalidArgument("top-k: k must be in [1, 1024]");
  if (max_len <= kWarpTkMax) {
    const unsigned grid = (unsigned)std::min<int64_t>(ceil_div(n_rows, kCandThreads / kWarp), (int64_t)kNumSMsB200 * 16);
    topk_segments_warp_kernel<<<grid, kCandThreads, 0, s>>>(SegmentRows{seg, scores}, n_rows, k, out_idx, out_score,
                                                            out_count);
  } else {
    const unsigned grid = (unsigned)std::min<int64_t>(n_rows, (int64_t)kNumSMsB200 * 8);
    topk_segments_kernel<<<grid, kTkThreads, 0, s>>>(SegmentRows{seg, scores}, n_rows, k, out_idx, out_score,
                                                     out_count);
  }
  count_launch();
  CUDA_CHECK(cudaGetLastError());
}

}  // namespace ials
