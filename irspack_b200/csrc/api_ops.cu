// Standalone tensor-core weighted Gram operators on host buffers (tests, parity tools).
#include <algorithm>
#include <vector>

#include "trainer.cuh"

using namespace ials;

namespace {

// The entries of a weighted Gram operator on the device: gathered row ids (optional), weights
// (optional) and the job bounds.
struct GramEntries {
  DeviceBuffer<int32_t> idx;
  DeviceBuffer<float> w;
  DeviceBuffer<int64_t> job_begin, job_end;

  void upload(const int32_t *idx_host, const float *w_host, int64_t m, const int64_t *jb, const int64_t *je,
              int64_t n_jobs) {
    if (idx_host) {
      idx.alloc(std::max<int64_t>(m, 1));
      CUDA_CHECK(cudaMemcpy(idx.get(), idx_host, sizeof(int32_t) * m, cudaMemcpyHostToDevice));
    }
    if (w_host) {
      w.alloc(std::max<int64_t>(m, 1));
      CUDA_CHECK(cudaMemcpy(w.get(), w_host, sizeof(float) * m, cudaMemcpyHostToDevice));
    }
    job_begin.alloc(n_jobs);
    job_end.alloc(n_jobs);
    CUDA_CHECK(cudaMemcpy(job_begin.get(), jb, sizeof(int64_t) * n_jobs, cudaMemcpyHostToDevice));
    CUDA_CHECK(cudaMemcpy(job_end.get(), je, sizeof(int64_t) * n_jobs, cudaMemcpyHostToDevice));
  }

  // An even split of the m entries into n_jobs jobs.
  void upload_even(const int32_t *idx_host, const float *w_host, int64_t m, int64_t n_jobs) {
    std::vector<int64_t> jb(n_jobs), je(n_jobs);
    const int64_t per = (m + n_jobs - 1) / n_jobs;
    for (int64_t j = 0; j < n_jobs; j++) {
      jb[j] = std::min(j * per, m);
      je[j] = std::min(jb[j] + per, m);
    }
    upload(idx_host, w_host, m, jb.data(), je.data(), n_jobs);
  }

  WGramArgs args(float bias) const {
    WGramArgs a{};
    a.indices = idx.get();
    a.weights = w.get();
    a.job_begin = job_begin.get();
    a.job_end = job_end.get();
    a.n_jobs = (int64_t)job_begin.size();
    a.bias = bias;
    return a;
  }
};

void check_entries(int64_t n, const int32_t *idx_host, const float *w_host, int64_t m) {
  require(m >= 0 && m <= kMaxGramEntries, "m must be in [0, 2^31 - 64]");
  if (idx_host)
    for (int64_t i = 0; i < m; i++) require(idx_host[i] >= 0 && idx_host[i] < n, "index out of range");
  if (w_host)
    for (int64_t i = 0; i < m; i++) require(w_host[i] >= 0.f, "weights must be non-negative");
}

}  // namespace

extern "C" {

// Standalone operator: G = sum_t w_t y_{i_t} y_{i_t}^T (and b = sum (bias + w_t) y_{i_t}) on the
// tensor cores, host buffers in and out.
int ials_weighted_gram(const float *Y_host, int64_t n, int64_t K, const int32_t *idx_host,
                       const float *w_host, int64_t m, int64_t n_jobs, float bias, int device,
                       float *G_host, float *b_host) {
  return guarded([&] {
    require(Y_host != nullptr && G_host != nullptr, "null pointer");
    require(n >= 0 && K >= 1 && K <= 128, "K must be in [1, 128]");
    require(n_jobs >= 1 && n_jobs <= 4096, "n_jobs must be in [1, 4096]");
    const bool gathered = idx_host != nullptr;
    if (!gathered) m = n;
    check_entries(n, idx_host, w_host, m);
    require_device(device);
    DeviceGuard g(device);
    const int ld = 128;
    cudaStream_t s = nullptr;
    DeviceBuffer<float> d_tmp, d_Y, d_W, d_b, d_G;
    GramEntries entries;
    DeviceSyncOnExit sync;
    d_tmp.alloc(std::max<int64_t>(n * K, 1));
    d_Y.alloc(std::max<int64_t>(n * ld, 1));
    CUDA_CHECK(cudaMemcpy(d_tmp.get(), Y_host, sizeof(float) * n * K, cudaMemcpyHostToDevice));
    launch_pad_copy(d_tmp.get(), n, (int)K, d_Y.get(), ld, s);
    entries.upload_even(gathered ? idx_host : nullptr, w_host, m, n_jobs);
    WGramArgs a = entries.args(bias);
    a.Y = d_Y.get();
    a.ld = ld;
    a.W = d_W.alloc(n_jobs * ld * ld);
    a.bpart = d_b.alloc(n_jobs * kWGramBParts * ld);
    d_G.alloc(ld * ld);
    launch_wgram(a, s);
    launch_wgram_reduce_sym(d_W.get(), (int)n_jobs, 1.0f, d_G.get(), s);
    CUDA_CHECK(cudaStreamSynchronize(s));
    rows_to_host(G_host, K, d_G.get(), ld, K);
    if (b_host) {
      std::vector<float> hb((size_t)n_jobs * kWGramBParts * ld);
      CUDA_CHECK(cudaMemcpy(hb.data(), d_b.get(), sizeof(float) * hb.size(), cudaMemcpyDeviceToHost));
      for (int64_t k = 0; k < K; k++) {
        float acc = 0.f;
        for (int64_t p = 0; p < n_jobs * kWGramBParts; p++) acc += hb[p * ld + k];
        b_host[k] = acc;
      }
    }
    CUDA_CHECK(cudaDeviceSynchronize());
  });
}

// Standalone operator for 256-column factors (K = 256 Cholesky, BASELINE configs[2]): the
// tensor-core launch of solve_cholesky_tensor (wgram256_kernel) on host buffers, its per-job
// W blocks assembled into G = sum w y y^T (256 x 256) and b = sum (bias + w) y.
int ials_weighted_gram256(const float *Y_host, int64_t n, int64_t K, const int32_t *idx_host,
                          const float *w_host, int64_t m, int64_t n_jobs, float bias, int device,
                          float *G_host, float *b_host) {
  return guarded([&] {
    require(Y_host != nullptr && G_host != nullptr && idx_host != nullptr, "null pointer");
    require(n >= 1 && K > 128 && K <= 256, "K must be in (128, 256]");
    require(n_jobs >= 1 && n_jobs <= 1024, "n_jobs must be in [1, 1024]");
    check_entries(n, idx_host, w_host, m);
    require_device(device);
    DeviceGuard g(device);
    const int ld = 256;
    const size_t blk = (size_t)n_jobs * 256 * 256, bsz = (size_t)n_jobs * kWGram256BParts * 256;
    cudaStream_t s = nullptr;
    DeviceBuffer<float> d_Y, d_ws;
    GramEntries entries;
    DeviceSyncOnExit sync;
    CUDA_CHECK(cudaMemset(d_Y.alloc(n * ld), 0, sizeof(float) * n * ld));
    rows_to_device(d_Y.get(), ld, Y_host, K, n);
    entries.upload_even(idx_host, w_host, m, n_jobs);
    WGramArgs a = entries.args(bias);
    a.ld = ld;
    a.Y = d_Y.get();
    a.W = d_ws.alloc(blk + bsz);
    a.bpart = a.W + blk;
    launch_wgram256(a, s);
    std::vector<float> h(blk + bsz);
    CUDA_CHECK(cudaMemcpy(h.data(), d_ws.get(), sizeof(float) * h.size(), cudaMemcpyDeviceToHost));
    std::vector<double> G((size_t)256 * 256, 0.0);
    for (int64_t j = 0; j < n_jobs; j++) {
      const float *W = h.data() + j * 65536;
      for (int r = 0; r < 256; r++)
        for (int c = 0; c < 256; c++) G[(size_t)r * 256 + c] += (double)W[r * 256 + c] + (double)W[c * 256 + r];
    }
    for (int64_t r = 0; r < K; r++)
      for (int64_t c = 0; c < K; c++) G_host[r * K + c] = (float)G[(size_t)r * 256 + c];
    if (b_host)
      for (int64_t k = 0; k < K; k++) {
        const float *bp = h.data() + blk + k;
        double acc = 0.0;
        for (int64_t q = 0; q < n_jobs * kWGram256BParts; q++) acc += bp[q * 256];
        b_host[k] = (float)acc;
      }
  });
}

// The same operators job by job, on explicit job bounds: job j takes the entries
// [job_begin[j], job_end[j]) of (idx, w) -- of the rows of Y when idx is null -- in one launch of
// wgram_kernel (K <= 128, row stride 128) or wgram256_kernel (K <= 256, row stride 256), and its own
// block comes back: G_jobs[j] = W_j + W_j^T (K x K) and b_jobs[j] = the sum of its producers'
// partials of (bias + w) y.  These are the blocks the trainer's solvers add up per row.
int ials_weighted_gram_jobs(const float *Y_host, int64_t n, int64_t K, const int32_t *idx_host,
                            const float *w_host, int64_t m, const int64_t *job_begin, const int64_t *job_end,
                            int64_t n_jobs, float bias, int device, float *G_jobs, float *b_jobs) {
  return guarded([&] {
    require(Y_host != nullptr && job_begin != nullptr && job_end != nullptr && G_jobs != nullptr,
            "null pointer");
    require(n >= 0 && K >= 1 && K <= 256, "K must be in [1, 256]");
    const bool wide = K > 128;
    require(n_jobs >= 1 && n_jobs <= (wide ? 1024 : 4096),
            wide ? "n_jobs must be in [1, 1024] for K > 128" : "n_jobs must be in [1, 4096]");
    if (idx_host == nullptr) m = n;
    check_entries(n, idx_host, w_host, m);
    for (int64_t j = 0; j < n_jobs; j++)
      require(job_begin[j] >= 0 && job_begin[j] <= job_end[j] && job_end[j] <= m,
              "job bounds must satisfy 0 <= begin <= end <= m");
    require_device(device);
    DeviceGuard g(device);
    const int ld = wide ? 256 : 128, parts = wide ? kWGram256BParts : kWGramBParts;
    const size_t blk = (size_t)ld * ld;
    cudaStream_t s = nullptr;
    DeviceBuffer<float> d_Y, d_W, d_b;
    GramEntries entries;
    DeviceSyncOnExit sync;
    CUDA_CHECK(cudaMemset(d_Y.alloc(std::max<int64_t>(n * ld, 1)), 0, sizeof(float) * std::max<int64_t>(n * ld, 1)));
    if (n) rows_to_device(d_Y.get(), ld, Y_host, K, n);
    entries.upload(idx_host, w_host, m, job_begin, job_end, n_jobs);
    WGramArgs a = entries.args(bias);
    a.Y = d_Y.get();
    a.ld = ld;
    a.W = d_W.alloc(n_jobs * blk);
    a.bpart = d_b.alloc(n_jobs * parts * ld);
    if (wide)
      launch_wgram256(a, s);
    else
      launch_wgram(a, s);
    std::vector<float> hW((size_t)n_jobs * blk), hb((size_t)n_jobs * parts * ld);
    CUDA_CHECK(cudaMemcpy(hW.data(), d_W.get(), sizeof(float) * hW.size(), cudaMemcpyDeviceToHost));
    CUDA_CHECK(cudaMemcpy(hb.data(), d_b.get(), sizeof(float) * hb.size(), cudaMemcpyDeviceToHost));
    for (int64_t j = 0; j < n_jobs; j++) {
      const float *W = hW.data() + j * blk;
      float *G = G_jobs + j * K * K;
      for (int64_t r = 0; r < K; r++)
        for (int64_t c = 0; c < K; c++) G[r * K + c] = W[r * ld + c] + W[c * ld + r];
      if (b_jobs)
        for (int64_t k = 0; k < K; k++) {
          double acc = 0.0;
          for (int p = 0; p < parts; p++) acc += hb[((size_t)j * parts + p) * ld + k];
          b_jobs[j * K + k] = (float)acc;
        }
    }
  });
}

}  // extern "C"
