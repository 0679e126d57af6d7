// K4 score block  S = user[b:e] item^T   (replaces IALSTrainer::user_scores,
//    /root/reference/cpp_source/als/IALSTrainer.hpp:942-984),
// K6 seen mask    S[mask.nonzero()] = -inf
//    (/root/reference/src/irspack/evaluation/evaluator.py:426-432),
// K5 top-k        first `k` of the candidates ordered by (-score, index)
//    (/root/reference/cpp_source/evaluator.cpp:324-355).
//
// v0: FP32 SIMT 128x128 register-tiled GEMM, a scatter kernel for the mask and a
// CTA-per-row threshold-filter top-k that orders 64-bit keys
// (order-preserving bits of -score) << 32 | index, i.e. exactly the reference's
// lexicographic pair comparison.
#include "topk.cuh"

namespace ials {
namespace {

constexpr int kTile = 128;
constexpr int kKc = 16;
constexpr int kThreads = 256;

__global__ void __launch_bounds__(kThreads)
score_tile_kernel(const float *__restrict__ A, int64_t n_rows, const float *__restrict__ B,
                  int64_t n_items, int ld, float *__restrict__ C, int64_t out_ld) {
  __shared__ __align__(16) float As[kKc][kTile + 4];
  __shared__ __align__(16) float Bs[kKc][kTile + 4];
  const int tid = threadIdx.x, tx = tid % 16, ty = tid / 16;
  const int64_t r0 = (int64_t)blockIdx.y * kTile, c0 = (int64_t)blockIdx.x * kTile;
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; i++)
#pragma unroll
    for (int j = 0; j < 8; j++) acc[i][j] = 0.f;

  for (int k0 = 0; k0 < ld; k0 += kKc) {
    // 128 rows x 16 k = 512 float4 per operand, 2 per thread, stored transposed
#pragma unroll
    for (int it = 0; it < 2; it++) {
      const int f = tid + it * kThreads;
      const int rr = f / (kKc / 4), kk = (f % (kKc / 4)) * 4;
      float4 va = make_float4(0.f, 0.f, 0.f, 0.f), vb = va;
      if (r0 + rr < n_rows) va = *reinterpret_cast<const float4 *>(A + (r0 + rr) * ld + k0 + kk);
      if (c0 + rr < n_items) vb = *reinterpret_cast<const float4 *>(B + (c0 + rr) * ld + k0 + kk);
      As[kk + 0][rr] = va.x; As[kk + 1][rr] = va.y; As[kk + 2][rr] = va.z; As[kk + 3][rr] = va.w;
      Bs[kk + 0][rr] = vb.x; Bs[kk + 1][rr] = vb.y; Bs[kk + 2][rr] = vb.z; Bs[kk + 3][rr] = vb.w;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < kKc; kk++) {
      float a[8], b[8];
      *reinterpret_cast<float4 *>(&a[0]) = *reinterpret_cast<const float4 *>(&As[kk][ty * 4]);
      *reinterpret_cast<float4 *>(&a[4]) = *reinterpret_cast<const float4 *>(&As[kk][64 + ty * 4]);
      *reinterpret_cast<float4 *>(&b[0]) = *reinterpret_cast<const float4 *>(&Bs[kk][tx * 4]);
      *reinterpret_cast<float4 *>(&b[4]) = *reinterpret_cast<const float4 *>(&Bs[kk][64 + tx * 4]);
#pragma unroll
      for (int i = 0; i < 8; i++)
#pragma unroll
        for (int j = 0; j < 8; j++) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
  const bool vec_ok = (out_ld % 4) == 0;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    const int64_t r = r0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
    if (r >= n_rows) continue;
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const int64_t c = c0 + h * 64 + tx * 4;
      float *dst = C + r * out_ld + c;
      if (vec_ok && c + 3 < n_items) {
        *reinterpret_cast<float4 *>(dst) =
            make_float4(acc[i][h * 4 + 0], acc[i][h * 4 + 1], acc[i][h * 4 + 2], acc[i][h * 4 + 3]);
      } else {
#pragma unroll
        for (int j = 0; j < 4; j++)
          if (c + j < n_items) dst[j] = acc[i][h * 4 + j];
      }
    }
  }
}

// One warp per user row of the mask CSR; stored zeros are skipped because
// scipy's `.nonzero()` drops them (evaluator.py:432).
__global__ void mask_rows_kernel(float *__restrict__ scores, int64_t out_ld,
                                 const int64_t *__restrict__ indptr,
                                 const int32_t *__restrict__ indices,
                                 const float *__restrict__ data, int64_t row0, int64_t n_rows,
                                 int64_t indptr_base) {
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / kWarp;
  const int lane = threadIdx.x % kWarp;
  if (warp >= n_rows) return;
  const int64_t s = indptr[row0 + warp] - indptr_base, e = indptr[row0 + warp + 1] - indptr_base;
  for (int64_t j = s + lane; j < e; j += kWarp)
    if (data == nullptr || data[j] != 0.f) scores[warp * out_ld + indices[j]] = -INFINITY;
}

// Allow-lists of retrieve_recommend_from_score (cpp_source/util.hpp:458-473): dst is -inf
// everywhere except at the allowed, in-range columns of each row, where it takes src.
// One warp per row; n_lists == 1 shares list 0 between all rows.
__global__ void fill_kernel(float *__restrict__ p, int64_t n, float v) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    p[i] = v;
}
__global__ void allow_rows_kernel(const float *__restrict__ src, float *__restrict__ dst, int64_t ld,
                                  const int64_t *__restrict__ indptr,
                                  const int64_t *__restrict__ indices, int64_t n_lists, int64_t row0,
                                  int64_t n_rows, int64_t n_items) {
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / kWarp;
  const int lane = threadIdx.x % kWarp;
  if (warp >= n_rows) return;
  const int64_t list = n_lists == 1 ? 0 : row0 + warp;
  const int64_t s = indptr[list], e = indptr[list + 1];
  for (int64_t j = s + lane; j < e; j += kWarp) {
    const int64_t c = indices[j];
    if (c >= 0 && c < n_items) dst[warp * ld + c] = src[warp * ld + c];
  }
}

// dense score rows: row r is scores[r * out_ld, + n_items), the column id is the position
struct DenseRows {
  const float *scores;
  int64_t out_ld, n_items;
  struct Row {
    const float *s;
    int64_t n;
    __device__ float score(int64_t j) const { return s[j]; }
    __device__ uint32_t id(int64_t j) const { return (uint32_t)j; }
  };
  __device__ Row row(int64_t r) const { return {scores + r * out_ld, n_items}; }
};

__global__ void __launch_bounds__(kTkThreads)
topk_rows_kernel(const float *__restrict__ scores, int64_t out_ld, int64_t n_rows, int64_t n_items,
                 int k, int32_t *__restrict__ out_idx, float *__restrict__ out_score,
                 int32_t *__restrict__ out_count) {
  topk_rows_body(DenseRows{scores, out_ld, n_items}, n_rows, k, out_idx, out_score, out_count);
}

}  // namespace

void launch_scores(const float *user_rows, int64_t n_rows, const float *item, int64_t n_items,
                   int ld, float *out, int64_t out_ld, cudaStream_t s) {
  if (n_rows == 0 || n_items == 0) return;
  dim3 grid((unsigned)ceil_div(n_items, kTile), (unsigned)ceil_div(n_rows, kTile));
  score_tile_kernel<<<grid, kThreads, 0, s>>>(user_rows, n_rows, item, n_items, ld, out, out_ld); count_launch();
  CUDA_CHECK(cudaGetLastError());
}

void launch_mask_rows(float *scores, int64_t out_ld, const int64_t *indptr, const int32_t *indices,
                      const float *data, int64_t row0, int64_t n_rows, int64_t indptr_base,
                      cudaStream_t s) {
  if (n_rows == 0) return;
  const int T = 256;
  mask_rows_kernel<<<(unsigned)ceil_div(n_rows * kWarp, T), T, 0, s>>>(
      scores, out_ld, indptr, indices, data, row0, n_rows, indptr_base); count_launch();
  CUDA_CHECK(cudaGetLastError());
}

void launch_allow_rows(const float *src, float *dst, int64_t ld, const int64_t *indptr,
                       const int64_t *indices, int64_t n_lists, int64_t row0, int64_t n_rows,
                       int64_t n_items, cudaStream_t s) {
  if (n_rows == 0) return;
  const int T = 256;
  const int64_t n = n_rows * ld;
  fill_kernel<<<(unsigned)std::min<int64_t>(ceil_div(n, T), (int64_t)kNumSMsB200 * 16), T, 0, s>>>(dst, n, -INFINITY);
  count_launch();
  allow_rows_kernel<<<(unsigned)ceil_div(n_rows * kWarp, T), T, 0, s>>>(src, dst, ld, indptr, indices, n_lists,
                                                                    row0, n_rows, n_items);
  count_launch();
  CUDA_CHECK(cudaGetLastError());
}

void launch_topk_rows(const float *scores, int64_t out_ld, int64_t n_rows, int64_t n_items, int k,
                      int32_t *out_idx, float *out_score, int32_t *out_count, cudaStream_t s) {
  if (n_rows == 0) return;
  if (k < 1 || k > kTkCap - kTkChunk) throw InvalidArgument("top-k: k must be in [1, 1024]");
  const unsigned grid = (unsigned)std::min<int64_t>(n_rows, (int64_t)kNumSMsB200 * 8);
  topk_rows_kernel<<<grid, kTkThreads, 0, s>>>(scores, out_ld, n_rows, n_items, k, out_idx,
                                               out_score, out_count); count_launch();
  CUDA_CHECK(cudaGetLastError());
}

}  // namespace ials
