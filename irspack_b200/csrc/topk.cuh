// CTA-per-row threshold-filter top-k (internal), shared by the dense rows of score.cu and the
// candidate segments of candidates.cu: the body is templated over how a row's scores and column ids
// are read, so each caller compiles to its own kernel without a branch on the other.
#pragma once
#include <cub/block/block_radix_sort.cuh>

#include "common.cuh"

namespace ials {

constexpr int kTkThreads = 256;
constexpr int kTkItems = 8;
constexpr int kTkCap = kTkThreads * kTkItems;  // 2048 candidate keys
constexpr int kTkChunk = 1024;                 // columns scanned between capacity checks

// Keeps the best k keys make_key(score, id) of rows [0, n_rows) (grid-stride over rows, one CTA per
// row), -inf scores dropped.  Rows::row(r) gives a view with the row's length n, score(j) and id(j).
// Writes out_idx / out_score [n_rows x k] (padded with -1 / -inf) and out_count [n_rows].
template <class Rows>
__device__ __forceinline__ void topk_rows_body(const Rows &rows, int64_t n_rows, int k, int32_t *__restrict__ out_idx,
                                               float *__restrict__ out_score, int32_t *__restrict__ out_count) {
  using Sort = cub::BlockRadixSort<unsigned long long, kTkThreads, kTkItems>;
  __shared__ typename Sort::TempStorage sort_tmp;
  __shared__ unsigned long long buf[kTkCap];
  __shared__ int cnt;
  __shared__ unsigned long long tau;
  const int tid = threadIdx.x;

  auto compact = [&]() {  // sort the candidates, keep the best k, tighten the threshold
    unsigned long long keys[kTkItems];
    const int n = cnt;
#pragma unroll
    for (int i = 0; i < kTkItems; i++) {
      const int p = tid * kTkItems + i;
      keys[i] = p < n ? buf[p] : ~0ull;
    }
    __syncthreads();
    Sort(sort_tmp).Sort(keys);
    __syncthreads();
#pragma unroll
    for (int i = 0; i < kTkItems; i++) buf[tid * kTkItems + i] = keys[i];
    __syncthreads();
    if (tid == 0) {
      if (n >= k) { cnt = k; tau = buf[k - 1]; }
    }
    __syncthreads();
  };

  for (int64_t row = blockIdx.x; row < n_rows; row += gridDim.x) {
    __syncthreads();
    if (tid == 0) { cnt = 0; tau = ~0ull; }
    __syncthreads();
    const auto src = rows.row(row);
    for (int64_t base = 0; base < src.n; base += kTkChunk) {
      const unsigned long long t = tau;
#pragma unroll
      for (int q = 0; q < kTkChunk / kTkThreads; q++) {
        const int64_t j = base + tid + q * kTkThreads;
        if (j < src.n) {
          const float sc = src.score(j);
          if (sc != -INFINITY) {
            const unsigned long long key = make_key(sc, src.id(j));
            if (key < t) buf[atomicAdd(&cnt, 1)] = key;
          }
        }
      }
      __syncthreads();
      const int settled = cnt;
      __syncthreads();  // every thread has read cnt before the next chunk's atomicAdd moves it
      if (settled > kTkCap - kTkChunk) compact();  // uniform
    }
    compact();
    const int n_out = min(cnt, k);
    for (int i = tid; i < k; i += kTkThreads) {
      const bool ok = i < n_out;
      out_idx[row * k + i] = ok ? (int32_t)(buf[i] & 0xffffffffu) : -1;
      if (out_score) out_score[row * k + i] = ok ? key_score(buf[i]) : -INFINITY;
    }
    if (tid == 0) out_count[row] = n_out;
  }
}

}  // namespace ials
