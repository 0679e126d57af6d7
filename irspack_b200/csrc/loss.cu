// iALS loss (replaces IALSTrainer::compute_loss without features,
// /root/reference/cpp_source/als/IALSTrainer.hpp:836-940):
//   loss = [ sum(P_user .* P_item) / alpha0
//            + sum_{(u,i) in S} (c p^2 - 2 (c + bias) p + c + bias)
//            + sum_u reg_u |x_u|^2 + sum_i reg_i |y_i|^2 ] / 2
// One warp per row; partial sums are accumulated in double (the reference
// accumulates in float; a scalar, so the extra precision is free).
#include "common.cuh"

namespace ials {
namespace {

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_sum_f(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// observed = 1: interaction terms + regulariser of `self` rows; 0: regulariser only
__global__ void loss_rows_kernel(const float *__restrict__ self, const float *__restrict__ other,
                                 int64_t n_rows, int64_t n_other, int ld,
                                 const int64_t *__restrict__ indptr,
                                 const int32_t *__restrict__ indices,
                                 const float *__restrict__ data, float alpha0, float reg, float nu,
                                 float bias, int observed, const float *__restrict__ prior,
                                 double *__restrict__ out) {
  const int lane = threadIdx.x % kWarp;
  const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / kWarp;
  const int64_t n_warps = (int64_t)gridDim.x * blockDim.x / kWarp;
  double total = 0.0;
  for (int64_t u = warp0; u < n_rows; u += n_warps) {
    const float *x = self + u * ld;
    const int64_t s = indptr[u], e = indptr[u + 1];
    float xx = 0.f;  // |x|^2, or |x - prior|^2 in the feature-aware model (:919-937)
    for (int k = lane; k < ld; k += kWarp) {
      const float d = prior ? x[k] - prior[u * ld + k] : x[k];
      xx = fmaf(d, d, xx);
    }
    xx = warp_sum_f(xx);
    const float reg_u = reg * powf(alpha0 * (float)n_other + (float)(e - s), nu);
    double row = (double)reg_u * (double)xx;
    if (observed) {
      for (int64_t j = s; j < e; j++) {
        const float *y = other + (int64_t)indices[j] * ld;
        float d = 0.f;
        for (int k = lane; k < ld; k += kWarp) d = fmaf(x[k], y[k], d);
        d = warp_sum_f(d);
        const float c = data[j];
        row += (double)(c * d * d - 2.f * (c + bias) * d + c + bias);
      }
    }
    total += row;
  }
  if (lane == 0 && total != 0.0) atomicAdd(out, total);
}

__global__ void loss_gram_kernel(const float *__restrict__ Pu, const float *__restrict__ Pi, int n,
                                 float alpha0, double *__restrict__ out) {
  double acc = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    acc += (double)Pu[i] * (double)Pi[i];
  acc = warp_sum_d(acc);
  if (threadIdx.x % kWarp == 0 && acc != 0.0) atomicAdd(out, acc / (double)alpha0);
}

__global__ void loss_halve_kernel(double *out) { *out *= 0.5; }

__global__ void loss_sumsq_kernel(const float *__restrict__ v, int64_t n, float scale, double *__restrict__ out) {
  double acc = 0.0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    acc += (double)v[i] * (double)v[i];
  acc = warp_sum_d(acc);
  if (threadIdx.x % kWarp == 0 && acc != 0.0) atomicAdd(out, (double)scale * acc);
}

}  // namespace

// The sum is left un-halved in *d_out: the caller adds the feature-weight ridge terms (if any) and
// calls launch_loss_halve.
void launch_loss(const float *user, const float *item, int64_t U, int64_t I, int K, int ld,
                 const DeviceCsr &X, const DeviceCsr &Xt, const float *Pu, const float *Pi,
                 float alpha0, float reg, float nu, float bias, const float *prior_u,
                 const float *prior_i, double *d_out, cudaStream_t s) {
  (void)K;
  CUDA_CHECK(cudaMemsetAsync(d_out, 0, sizeof(double), s));
  if (alpha0 != 0.f) loss_gram_kernel<<<32, 256, 0, s>>>(Pu, Pi, ld * ld, alpha0, d_out); count_launch();
  const int T = 256;
  if (U > 0)
    loss_rows_kernel<<<(unsigned)std::min<int64_t>(ceil_div(U * kWarp, T), kNumSMsB200 * 16), T, 0,
                       s>>>(user, item, U, I, ld, X.indptr.get(), X.indices.get(), X.data.get(), alpha0, reg, nu,
                            bias, 1, prior_u, d_out); count_launch();
  if (I > 0)
    loss_rows_kernel<<<(unsigned)std::min<int64_t>(ceil_div(I * kWarp, T), kNumSMsB200 * 16), T, 0,
                       s>>>(item, user, I, U, ld, Xt.indptr.get(), Xt.indices.get(), Xt.data.get(), alpha0, reg, nu,
                            bias, 0, prior_i, d_out); count_launch();
  CUDA_CHECK(cudaGetLastError());
}

void launch_loss_shard(const float *user, const float *item, int64_t U, int64_t I, int ld, const DeviceCsr &X,
                       const DeviceCsr &Xt, const float *Pu, const float *Pi, float alpha0, float reg, float nu,
                       float bias, const float *prior_u, const float *prior_i, double *d_out, cudaStream_t s) {
  CUDA_CHECK(cudaMemsetAsync(d_out, 0, sizeof(double), s));
  if (Pu != nullptr && alpha0 != 0.f) {
    loss_gram_kernel<<<32, 256, 0, s>>>(Pu, Pi, ld * ld, alpha0, d_out);
    count_launch();
  }
  const int T = 256;
  if (X.n_rows > 0) {
    loss_rows_kernel<<<(unsigned)std::min<int64_t>(ceil_div(X.n_rows * kWarp, T), kNumSMsB200 * 16), T, 0, s>>>(
        user + X.row_base * ld, item, X.n_rows, I, ld, X.indptr.get(), X.indices.get(), X.data.get(), alpha0, reg,
        nu, bias, 1, prior_u, d_out);
    count_launch();
  }
  if (Xt.n_rows > 0) {
    loss_rows_kernel<<<(unsigned)std::min<int64_t>(ceil_div(Xt.n_rows * kWarp, T), kNumSMsB200 * 16), T, 0, s>>>(
        item + Xt.row_base * ld, user, Xt.n_rows, U, ld, Xt.indptr.get(), Xt.indices.get(), Xt.data.get(), alpha0,
        reg, nu, bias, 0, prior_i, d_out);
    count_launch();
  }
  CUDA_CHECK(cudaGetLastError());
}

// *d_out += scale * sum v^2   (lambda |W|^2 of the feature weights, :929, :939)
void launch_loss_add_sumsq(const float *v, int64_t n, float scale, double *d_out, cudaStream_t s) {
  if (n <= 0) return;
  loss_sumsq_kernel<<<32, 256, 0, s>>>(v, n, scale, d_out); count_launch();
  CUDA_CHECK(cudaGetLastError());
}

void launch_loss_halve(double *d_out, cudaStream_t s) {
  loss_halve_kernel<<<1, 1, 0, s>>>(d_out); count_launch();
  CUDA_CHECK(cudaGetLastError());
}

}  // namespace ials
