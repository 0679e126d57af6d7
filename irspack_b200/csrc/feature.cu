// Feature-aware iALS, the parts around the row solves (replaces, on the device,
// /root/reference/cpp_source/als/IALSTrainer.hpp: feature_times_weight :696-702,
// initialize_feature_weight_cache :1083-1132, solve_feature_weight :1134-1180):
//
//   prior      = F W                                   (n x ld; the b of a row starts from reg_u * prior_u)
//   row weight = compute_reg(nnz_row)                  (cached with the Gram)
//   ridge      W = (F^T D F + lambda I)^-1 F^T D X     D = diag(row weights), X = the side's factors
//
// F is dense row-major or CSR.  This is the SURVEY 8 f4 "after that" row: plain kernels (a warp per
// feature row, fp32 atomics for the two F^T products, a one-CTA Cholesky of the n_cols x n_cols
// Gram that is computed once per trainer, a thread per factor column for the two triangular
// solves) -- correct and on the device, not tuned.
#include "common.cuh"

namespace ials {
namespace {

constexpr int kFThreads = 256;

// visit the stored entries (f, v) of feature row r
template <class Fn>
__device__ __forceinline__ void for_row(const FeatureDev &F, int64_t r, Fn &&fn) {
  if (F.dense) {
    const float *row = F.dense + r * F.n_cols;
    for (int64_t f = 0; f < F.n_cols; f++) fn(f, row[f]);
  } else {
    for (int64_t p = F.indptr[r]; p < F.indptr[r + 1]; p++) fn((int64_t)F.indices[p], F.data[p]);
  }
}

__global__ void __launch_bounds__(kFThreads) feature_prior_kernel(FeatureDev F, const float *__restrict__ W,
                                                                   int ld, float *__restrict__ out) {
  const int lane = threadIdx.x % kWarp;
  const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / kWarp;
  const int64_t n_warps = (int64_t)gridDim.x * blockDim.x / kWarp;
  for (int64_t r = warp0; r < F.n_rows; r += n_warps) {
    for (int c0 = 0; c0 < ld; c0 += 4 * kWarp) {  // 128 columns per sweep, 4 per lane
      float acc[4] = {0.f, 0.f, 0.f, 0.f};
      for_row(F, r, [&](int64_t f, float v) {
        const float *w = W + f * ld + c0 + lane;
#pragma unroll
        for (int j = 0; j < 4; j++)
          if (c0 + lane + 32 * j < ld) acc[j] = fmaf(v, w[32 * j], acc[j]);
      });
#pragma unroll
      for (int j = 0; j < 4; j++)
        if (c0 + lane + 32 * j < ld) out[r * ld + c0 + lane + 32 * j] = acc[j];
    }
  }
}

__global__ void feature_row_weights_kernel(const int64_t *__restrict__ indptr, int64_t n_rows, int64_t n_other,
                                           float alpha0, float reg, float nu, float *__restrict__ rw) {
  const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (r >= n_rows) return;
  rw[r] = reg * powf(alpha0 * (float)n_other + (float)(indptr[r + 1] - indptr[r]), nu);
}

// G += sum_r rw_r F_r^T F_r  (both triangles; a warp per row, lanes over the second index)
__global__ void __launch_bounds__(kFThreads) feature_gram_kernel(FeatureDev F, const float *__restrict__ rw,
                                                                  float *__restrict__ G) {
  const int lane = threadIdx.x % kWarp;
  const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / kWarp;
  const int64_t n_warps = (int64_t)gridDim.x * blockDim.x / kWarp;
  const int64_t n = F.n_cols;
  for (int64_t r = warp0; r < F.n_rows; r += n_warps) {
    const float w = rw[r];
    if (F.dense) {
      const float *row = F.dense + r * n;
      for (int64_t f = 0; f < n; f++) {
        const float wf = w * row[f];
        if (wf == 0.f) continue;
        for (int64_t g = lane; g < n; g += kWarp) {
          const float v = wf * row[g];
          if (v != 0.f) atomicAdd(&G[f * n + g], v);
        }
      }
    } else {
      const int64_t s = F.indptr[r], e = F.indptr[r + 1];
      for (int64_t p = s; p < e; p++) {
        const float wf = w * F.data[p];
        const int64_t f = F.indices[p];
        for (int64_t q = s + lane; q < e; q += kWarp) atomicAdd(&G[f * n + F.indices[q]], wf * F.data[q]);
      }
    }
  }
}

__global__ void feature_add_diag_kernel(float *G, int64_t n, float lambda) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) G[i * n + i] += lambda;
}

// In-place Cholesky G = L L^T (lower triangle of the row-major matrix), one CTA; Eigen's LLT rule:
// a pivot that is not positive fails ("Feature ridge Cholesky decomposition failed.").
__global__ void __launch_bounds__(1024) feature_llt_kernel(float *G, int n, int *fail) {
  __shared__ float s_d;
  __shared__ int s_bad;
  const int tid = threadIdx.x, T = blockDim.x;
  if (tid == 0) s_bad = 0;
  for (int k = 0; k < n; k++) {
    __syncthreads();
    if (tid == 0) {
      const float d = G[(size_t)k * n + k];
      if (!(d > 0.f)) s_bad = 1;
      s_d = sqrtf(d);
      G[(size_t)k * n + k] = s_d;
    }
    __syncthreads();
    if (s_bad) break;
    const float inv = 1.0f / s_d;
    for (int i = k + 1 + tid; i < n; i += T) G[(size_t)i * n + k] *= inv;
    __syncthreads();
    const int m = n - k - 1;
    for (int64_t e = tid; e < (int64_t)m * m; e += T) {
      const int i = k + 1 + (int)(e / m), j = k + 1 + (int)(e % m);
      if (j <= i) G[(size_t)i * n + j] = fmaf(-G[(size_t)i * n + k], G[(size_t)j * n + k], G[(size_t)i * n + j]);
    }
  }
  __syncthreads();
  if (tid == 0 && s_bad) atomicExch(fail, 1);
}

// R += sum_r rw_r F_r^T X_r   (R [n_cols x ld]; a warp per row, 4 columns per lane and sweep)
__global__ void __launch_bounds__(kFThreads) feature_rhs_kernel(FeatureDev F, const float *__restrict__ rw,
                                                                 const float *__restrict__ X, int ld,
                                                                 float *__restrict__ R) {
  const int lane = threadIdx.x % kWarp;
  const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / kWarp;
  const int64_t n_warps = (int64_t)gridDim.x * blockDim.x / kWarp;
  for (int64_t r = warp0; r < F.n_rows; r += n_warps) {
    const float w = rw[r];
    for (int c = lane; c < ld; c += kWarp) {
      const float wx = w * X[r * ld + c];
      if (wx == 0.f) continue;
      for_row(F, r, [&](int64_t f, float v) {
        if (v != 0.f) atomicAdd(&R[f * ld + c], v * wx);
      });
    }
  }
}

// W = (L L^T)^-1 R in place, a thread per column of R: forward then backward substitution.
__global__ void feature_solve_kernel(const float *__restrict__ L, int n, float *__restrict__ R, int ld,
                                     int *fail) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= ld) return;
  for (int i = 0; i < n; i++) {  // L y = r
    float v = R[(size_t)i * ld + c];
    const float *Li = L + (size_t)i * n;
    for (int j = 0; j < i; j++) v = fmaf(-Li[j], R[(size_t)j * ld + c], v);
    R[(size_t)i * ld + c] = v / Li[i];
  }
  bool finite = true;
  for (int i = n - 1; i >= 0; i--) {  // L^T w = y
    float v = R[(size_t)i * ld + c];
    for (int j = i + 1; j < n; j++) v = fmaf(-L[(size_t)j * n + i], R[(size_t)j * ld + c], v);
    v /= L[(size_t)i * n + i];
    R[(size_t)i * ld + c] = v;
    finite = finite && isfinite(v);
  }
  if (!finite) atomicExch(fail, 1);
}

unsigned warp_grid(int64_t n_rows) {
  return (unsigned)std::max<int64_t>(1, std::min<int64_t>(ceil_div(n_rows * kWarp, kFThreads), kNumSMsB200 * 8));
}

}  // namespace

void launch_feature_prior(const FeatureDev &F, const float *W, int ld, float *out, cudaStream_t s) {
  if (F.n_rows <= 0) return;
  feature_prior_kernel<<<warp_grid(F.n_rows), kFThreads, 0, s>>>(F, W, ld, out);
  count_launch();
  CUDA_CHECK(cudaGetLastError());
}

void launch_feature_row_weights(const int64_t *indptr, int64_t n_rows, int64_t n_other, float alpha0,
                                float reg, float nu, float *rw, cudaStream_t s) {
  if (n_rows <= 0) return;
  feature_row_weights_kernel<<<(unsigned)ceil_div(n_rows, 256), 256, 0, s>>>(indptr, n_rows, n_other, alpha0,
                                                                             reg, nu, rw);
  count_launch();
  CUDA_CHECK(cudaGetLastError());
}

void launch_feature_gram(const FeatureDev &F, const float *rw, float *G, cudaStream_t s) {
  const int64_t n = F.n_cols;
  if (n <= 0) return;
  CUDA_CHECK(cudaMemsetAsync(G, 0, sizeof(float) * n * n, s));
  if (F.n_rows > 0) {
    feature_gram_kernel<<<warp_grid(F.n_rows), kFThreads, 0, s>>>(F, rw, G);
    count_launch();
  }
  CUDA_CHECK(cudaGetLastError());
}

void launch_feature_llt(float *G, int64_t n, float lambda, int *fail, cudaStream_t s) {
  if (n <= 0) return;
  feature_add_diag_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, s>>>(G, n, lambda);
  count_launch();
  feature_llt_kernel<<<1, 1024, 0, s>>>(G, (int)n, fail);
  count_launch();
  CUDA_CHECK(cudaGetLastError());
}

void launch_feature_gram_llt(const FeatureDev &F, const float *rw, float lambda, float *G, int *fail,
                             cudaStream_t s) {
  launch_feature_gram(F, rw, G, s);
  launch_feature_llt(G, F.n_cols, lambda, fail, s);
}

void launch_feature_rhs(const FeatureDev &F, const float *rw, const float *X, int ld, float *R, cudaStream_t s) {
  const int64_t n = F.n_cols;
  if (n <= 0) return;
  CUDA_CHECK(cudaMemsetAsync(R, 0, sizeof(float) * n * ld, s));
  if (F.n_rows > 0) {
    feature_rhs_kernel<<<warp_grid(F.n_rows), kFThreads, 0, s>>>(F, rw, X, ld, R);
    count_launch();
  }
  CUDA_CHECK(cudaGetLastError());
}

void launch_feature_solve(const float *L, int64_t n, float *R, int ld, int *fail, cudaStream_t s) {
  if (n <= 0) return;
  feature_solve_kernel<<<(unsigned)ceil_div(ld, 64), 64, 0, s>>>(L, (int)n, R, ld, fail);
  count_launch();
  CUDA_CHECK(cudaGetLastError());
}

void launch_feature_ridge_solve(const FeatureDev &F, const float *rw, const float *X, int ld,
                                const float *L, float *R, int *fail, cudaStream_t s) {
  launch_feature_rhs(F, rw, X, ld, R, s);
  launch_feature_solve(L, F.n_cols, R, ld, fail, s);
}

}  // namespace ials
