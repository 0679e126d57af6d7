// CSR plumbing on the device: X^T construction (the reference does
// `X_t(X.transpose())` + makeCompressed on the host, IALSTrainer.hpp:713-716),
// the degree-sorted row schedule, and padded <-> dense factor copies.
#include <cub/cub.cuh>

#include <vector>

#include "common.cuh"

namespace ials {

namespace {

// row id of every stored element: one warp per row, lanes stride the row.
__global__ void expand_rows_kernel(const int64_t *__restrict__ indptr, int64_t n_rows,
                                   int32_t *__restrict__ row_of) {
  int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / kWarp;
  int lane = threadIdx.x % kWarp;
  int64_t n_warps = (int64_t)gridDim.x * blockDim.x / kWarp;
  for (int64_t r = warp; r < n_rows; r += n_warps) {
    int64_t s = indptr[r], e = indptr[r + 1];
    for (int64_t j = s + lane; j < e; j += kWarp) row_of[j] = (int32_t)r;
  }
}

__global__ void iota_kernel(uint32_t *p, int64_t n) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) p[i] = (uint32_t)i;
}

__global__ void gather_transposed_kernel(const uint32_t *__restrict__ perm,
                                         const int32_t *__restrict__ row_of,
                                         const float *__restrict__ data, int64_t nnz,
                                         int32_t *__restrict__ indices_t,
                                         float *__restrict__ data_t) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < nnz) {
    uint32_t p = perm[i];
    indices_t[i] = row_of[p];
    data_t[i] = data[p];
  }
}

// indptr_t[c] = first position in the column-sorted key array with key >= c.
__global__ void lower_bound_kernel(const int32_t *__restrict__ sorted_cols, int64_t nnz,
                                   int64_t n_cols, int64_t *__restrict__ indptr_t) {
  int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (c > n_cols) return;
  int64_t lo = 0, hi = nnz;
  while (lo < hi) {
    int64_t mid = (lo + hi) >> 1;
    if ((int64_t)sorted_cols[mid] < c) lo = mid + 1; else hi = mid;
  }
  indptr_t[c] = lo;
}

__global__ void degree_kernel(const int64_t *__restrict__ indptr, int64_t n_rows,
                              uint32_t *__restrict__ deg, uint32_t *__restrict__ ids) {
  int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (r < n_rows) {
    deg[r] = (uint32_t)(indptr[r + 1] - indptr[r]);
    ids[r] = (uint32_t)r;
  }
}

__global__ void pad_copy_kernel(const float *__restrict__ src, int64_t n_rows, int K,
                                float *__restrict__ dst, int ld) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  int64_t total = n_rows * ld;
  if (i < total) {
    int64_t r = i / ld;
    int k = (int)(i - r * ld);
    dst[i] = k < K ? src[r * K + k] : 0.f;
  }
}

// dst[r] = src[rows[r]] for factor rows of `ld` floats (ld % 4 == 0): one float4 per thread
__global__ void gather_rows_kernel(const float *__restrict__ src, int ld, const int64_t *__restrict__ rows,
                                   int64_t n_rows, float *__restrict__ dst) {
  const int per = ld >> 2;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_rows * per) return;
  const int64_t r = i / per;
  const int c = (int)(i - r * per);
  reinterpret_cast<float4 *>(dst + r * ld)[c] = reinterpret_cast<const float4 *>(src + rows[r] * ld)[c];
}

// dst[r] = src[r] / |src[r]| (rows of `ld` floats, ld % 4 == 0; a row of norm 0 stays 0): one warp per
// row, the sum of squares in float64 so that neither tiny nor huge rows lose their direction
__global__ void normalize_rows_kernel(const float *__restrict__ src, int64_t n_rows, int ld, float *__restrict__ dst) {
  const int64_t r = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / kWarp;
  const int lane = threadIdx.x % kWarp;
  if (r >= n_rows) return;
  const float4 *row = reinterpret_cast<const float4 *>(src + r * ld);
  double ss = 0.0;
  for (int c = lane; c < (ld >> 2); c += kWarp) {
    const float4 v = row[c];
    ss += (double)v.x * v.x + (double)v.y * v.y + (double)v.z * v.z + (double)v.w * v.w;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  const double inv = ss > 0.0 ? 1.0 / sqrt(ss) : 0.0;
  float4 *out = reinterpret_cast<float4 *>(dst + r * ld);
  for (int c = lane; c < (ld >> 2); c += kWarp) {
    const float4 v = row[c];
    out[c] = make_float4((float)(v.x * inv), (float)(v.y * inv), (float)(v.z * inv), (float)(v.w * inv));
  }
}

// The CSR whose row i lists column i alone: indptr[i] = i (i <= n), indices[i] = i (i < n)
__global__ void self_mask_kernel(int64_t *__restrict__ indptr, int32_t *__restrict__ indices, int64_t n) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i <= n) indptr[i] = i;
  if (i < n) indices[i] = (int32_t)i;
}

__global__ void unpad_copy_kernel(const float *__restrict__ src, int64_t n_rows, int K, int ld,
                                  float *__restrict__ dst) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  int64_t total = n_rows * K;
  if (i < total) {
    int64_t r = i / K;
    int k = (int)(i - r * K);
    dst[i] = src[r * ld + k];
  }
}

__device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

// Counter-based N(0, stdev) fill (Box-Muller on splitmix64 bits); used only for
// factor matrices too large for the reference's serial host RNG.
__global__ void init_normal_kernel(float *__restrict__ dst, int64_t n_rows, int K, int ld,
                                   float stdev, uint64_t seed) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  int64_t total = n_rows * ld;
  if (i < total) {
    int k = (int)(i % ld);
    float v = 0.f;
    if (k < K) {
      uint64_t h = splitmix64(seed ^ splitmix64((uint64_t)i));
      float u1 = ((uint32_t)(h >> 40) + 1) * (1.0f / 16777217.0f);
      float u2 = (uint32_t)((h >> 8) & 0xFFFFFF) * (1.0f / 16777216.0f);
      v = stdev * sqrtf(-2.f * logf(u1)) * cospif(2.f * u2);
    }
    dst[i] = v;
  }
}

int bits_for(int64_t n) {
  int b = 1;
  while (b < 32 && (1ll << b) < n) b++;
  return b;
}

}  // namespace

void build_transpose(const DeviceCsr &X, DeviceCsr &Xt, cudaStream_t s) {
  Xt.n_rows = X.n_cols;
  Xt.n_cols = X.n_rows;
  Xt.nnz = X.nnz;
  Xt.indptr.alloc(Xt.n_rows + 1);
  Xt.indices.alloc(std::max<int64_t>(X.nnz, 1));
  Xt.data.alloc(std::max<int64_t>(X.nnz, 1));
  const int64_t nnz = X.nnz;
  if (nnz == 0) {
    CUDA_CHECK(cudaMemsetAsync(Xt.indptr.get(), 0, sizeof(int64_t) * (Xt.n_rows + 1), s));
    return;
  }
  DeviceBuffer<int32_t> row_of, cols_sorted;
  DeviceBuffer<uint32_t> perm_in, perm_out;
  DeviceBuffer<char> tmp;
  StreamSyncOnExit sync{s};
  row_of.alloc(nnz);
  cols_sorted.alloc(nnz);
  perm_in.alloc(nnz);
  perm_out.alloc(nnz);
  const int T = 256;
  expand_rows_kernel<<<(unsigned)std::min<int64_t>(ceil_div(X.n_rows * kWarp, T), 65535 * 8), T, 0,
                       s>>>(X.indptr.get(), X.n_rows, row_of.get()); count_launch();
  iota_kernel<<<(unsigned)ceil_div(nnz, T), T, 0, s>>>(perm_in.get(), nnz); count_launch();
  // stable LSD radix sort by column keeps rows ascending inside each column
  size_t tmp_bytes = 0;
  const int end_bit = bits_for(X.n_cols);
  CUDA_CHECK(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, X.indices.get(), cols_sorted.get(), perm_in.get(),
                                             perm_out.get(), nnz, 0, end_bit, s));
  tmp.alloc(tmp_bytes);
  CUDA_CHECK(cub::DeviceRadixSort::SortPairs(tmp.get(), tmp_bytes, X.indices.get(), cols_sorted.get(), perm_in.get(),
                                             perm_out.get(), nnz, 0, end_bit, s));
  gather_transposed_kernel<<<(unsigned)ceil_div(nnz, T), T, 0, s>>>(perm_out.get(), row_of.get(), X.data.get(), nnz,
                                                                    Xt.indices.get(), Xt.data.get()); count_launch();
  lower_bound_kernel<<<(unsigned)ceil_div(Xt.n_rows + 1, T), T, 0, s>>>(cols_sorted.get(), nnz,
                                                                        Xt.n_rows, Xt.indptr.get()); count_launch();
  CUDA_CHECK(cudaGetLastError());
  CUDA_CHECK(cudaStreamSynchronize(s));
}

void build_row_order(DeviceCsr &X, cudaStream_t s) {
  const int64_t n = X.n_rows;
  X.order.alloc(std::max<int64_t>(n, 1));
  X.max_degree = 0;
  if (n == 0) return;
  DeviceBuffer<uint32_t> deg, deg_sorted, ids;
  DeviceBuffer<char> tmp;
  StreamSyncOnExit sync{s};
  deg.alloc(n);
  deg_sorted.alloc(n);
  ids.alloc(n);
  const int T = 256;
  degree_kernel<<<(unsigned)ceil_div(n, T), T, 0, s>>>(X.indptr.get(), n, deg.get(), ids.get()); count_launch();
  size_t tmp_bytes = 0;
  CUDA_CHECK(cub::DeviceRadixSort::SortPairsDescending(nullptr, tmp_bytes, deg.get(), deg_sorted.get(), ids.get(),
                                                       (uint32_t *)X.order.get(), n, 0, 32, s));
  tmp.alloc(tmp_bytes);
  CUDA_CHECK(cub::DeviceRadixSort::SortPairsDescending(tmp.get(), tmp_bytes, deg.get(), deg_sorted.get(), ids.get(),
                                                       (uint32_t *)X.order.get(), n, 0, 32, s));
  uint32_t maxdeg = 0;
  CUDA_CHECK(cudaMemcpyAsync(&maxdeg, deg_sorted.get(), sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  CUDA_CHECK(cudaStreamSynchronize(s));
  X.max_degree = maxdeg;
}

// Some stored value < 0 (or NaN)?  The rows of such a matrix all take the light path.
bool csr_has_negative(const DeviceCsr &X, cudaStream_t s) {
  if (X.nnz == 0) return false;
  DeviceBuffer<float> d_min;
  DeviceBuffer<char> tmp;
  StreamSyncOnExit sync{s};
  size_t tmp_bytes = 0;
  d_min.alloc(1);
  CUDA_CHECK(cub::DeviceReduce::Min(nullptr, tmp_bytes, X.data.get(), d_min.get(), X.nnz, s));
  tmp.alloc(tmp_bytes);
  CUDA_CHECK(cub::DeviceReduce::Min(tmp.get(), tmp_bytes, X.data.get(), d_min.get(), X.nnz, s));
  float h_min = 0.f;
  CUDA_CHECK(cudaMemcpyAsync(&h_min, d_min.get(), sizeof(float), cudaMemcpyDeviceToHost, s));
  CUDA_CHECK(cudaStreamSynchronize(s));
  return !(h_min >= 0.f);
}

// Host-side planning (once per matrix): which rows go to the tensor-core path and how
// their neighbour lists are cut into jobs.
void build_heavy_plan(const DeviceCsr &X, int64_t threshold, int64_t job_len, JobPlan &plan, cudaStream_t s) {
  plan = JobPlan{};
  const int64_t n = X.n_rows;
  if (n == 0 || X.order.get() == nullptr) return;
  std::vector<int64_t> indptr(n + 1);
  std::vector<int32_t> order(n);
  CUDA_CHECK(cudaMemcpyAsync(indptr.data(), X.indptr.get(), sizeof(int64_t) * (n + 1), cudaMemcpyDeviceToHost, s));
  CUDA_CHECK(cudaMemcpyAsync(order.data(), X.order.get(), sizeof(int32_t) * n, cudaMemcpyDeviceToHost, s));
  CUDA_CHECK(cudaStreamSynchronize(s));
  std::vector<int64_t> jb, je;
  std::vector<int32_t> first;
  int64_t h = 0;
  for (; h < n; h++) {  // `order` is sorted by descending degree
    const int64_t u = order[h];
    const int64_t b = indptr[u], e = indptr[u + 1];
    if (e - b <= threshold) break;
    first.push_back((int32_t)jb.size());
    plan.nnz_heavy += e - b;
    const int64_t pieces = ceil_div(e - b, job_len);
    const int64_t per = round_up(ceil_div(e - b, pieces), 32);  // whole pipeline stages
    for (int64_t p = b; p < e; p += per) {
      jb.push_back(p);
      je.push_back(std::min(p + per, e));
    }
  }
  first.push_back((int32_t)jb.size());
  plan.n_heavy = h;
  plan.n_jobs = (int64_t)jb.size();
  if (plan.n_heavy == 0) return;
  plan.job_begin.alloc(plan.n_jobs);
  plan.job_end.alloc(plan.n_jobs);
  plan.heavy_first_job.alloc(first.size());
  CUDA_CHECK(cudaMemcpy(plan.job_begin.get(), jb.data(), sizeof(int64_t) * plan.n_jobs, cudaMemcpyHostToDevice));
  CUDA_CHECK(cudaMemcpy(plan.job_end.get(), je.data(), sizeof(int64_t) * plan.n_jobs, cudaMemcpyHostToDevice));
  CUDA_CHECK(cudaMemcpy(plan.heavy_first_job.get(), first.data(), sizeof(int32_t) * first.size(),
                        cudaMemcpyHostToDevice));
}

void launch_gather_rows(const float *src, int ld, const int64_t *rows, int64_t n_rows, float *dst,
                        cudaStream_t s) {
  if (n_rows == 0) return;
  const int64_t total = n_rows * (ld >> 2);
  gather_rows_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, s>>>(src, ld, rows, n_rows, dst); count_launch();
  CUDA_CHECK(cudaGetLastError());
}

void launch_pad_copy(const float *src, int64_t n_rows, int K, float *dst, int ld, cudaStream_t s) {
  int64_t total = n_rows * ld;
  if (total == 0) return;
  pad_copy_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, s>>>(src, n_rows, K, dst, ld); count_launch();
  CUDA_CHECK(cudaGetLastError());
}

void launch_unpad_copy(const float *src, int64_t n_rows, int K, int ld, float *dst,
                       cudaStream_t s) {
  int64_t total = n_rows * K;
  if (total == 0) return;
  unpad_copy_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, s>>>(src, n_rows, K, ld, dst); count_launch();
  CUDA_CHECK(cudaGetLastError());
}

void launch_normalize_rows(const float *src, int64_t n_rows, int ld, float *dst, cudaStream_t s) {
  if (n_rows == 0) return;
  normalize_rows_kernel<<<(unsigned)ceil_div(n_rows * kWarp, 256), 256, 0, s>>>(src, n_rows, ld, dst); count_launch();
  CUDA_CHECK(cudaGetLastError());
}

void launch_self_mask(int64_t *indptr, int32_t *indices, int64_t n, cudaStream_t s) {
  self_mask_kernel<<<(unsigned)ceil_div(n + 1, 256), 256, 0, s>>>(indptr, indices, n); count_launch();
  CUDA_CHECK(cudaGetLastError());
}

void launch_init_normal(float *dst, int64_t n_rows, int K, int ld, float stdev, uint64_t seed,
                        cudaStream_t s) {
  int64_t total = n_rows * ld;
  if (total == 0) return;
  init_normal_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, s>>>(dst, n_rows, K, ld, stdev,
                                                                   seed); count_launch();
  CUDA_CHECK(cudaGetLastError());
}

}  // namespace ials
