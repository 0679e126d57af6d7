// Shared declarations of the B200-native iALS library (internal; the public
// surface is include/ials_b200.h).
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <stdint.h>
#include <utility>

#include <stdexcept>
#include <string>

#include "../../include/ials_b200.h"

namespace ials {

constexpr int kWarp = 32;
constexpr int kNumSMsB200 = 148;

// Device-side failure flags, one int each, checked after a half-epoch
// (the reference throws from its workers: IALSTrainer.hpp:249-254, 317-323).
enum ErrFlag : int {
  kErrCgSingular = 0, kErrCholDecomp = 1, kErrCholSolve = 2, kErrInternal = 3,
  kErrFeatureLlt = 4, kErrFeatureSolve = 5,  // feature ridge (IALSTrainer.hpp:1107, 1171)
  kNumErrFlags = 6
};

struct CudaError : std::runtime_error {
  using std::runtime_error::runtime_error;
};
struct InvalidArgument : std::invalid_argument {
  using std::invalid_argument::invalid_argument;
};
struct NotImplemented : std::runtime_error {
  using std::runtime_error::runtime_error;
};

inline void cuda_check(cudaError_t e, const char *what, const char *file, int line) {
  if (e != cudaSuccess) {
    throw CudaError(std::string("CUDA error: ") + cudaGetErrorString(e) + " in " + what + " (" +
                    file + ":" + std::to_string(line) + ")");
  }
}
#define CUDA_CHECK(x) ::ials::cuda_check((x), #x, __FILE__, __LINE__)

// Function attributes (cudaFuncSetAttribute) belong to the current device's context: a process
// that drives several devices must set them once per device, not once per process.
struct PerDeviceOnce {
  std::atomic<unsigned long long> done{0};
  template <class F>
  void run(F &&f) {
    int dev = 0;
    CUDA_CHECK(cudaGetDevice(&dev));
    const unsigned long long bit = 1ull << (dev & 63);
    if (done.load(std::memory_order_acquire) & bit) return;
    f();  // setting an attribute twice (two threads racing here) is harmless
    done.fetch_or(bit, std::memory_order_release);
  }
};

// Owning handles of device memory (and of the one pinned host array, the step_io flag source).
// Each alloc() is one plain cudaMalloc and each release one cudaFree: allocation timing is part of
// what the benchmarks measure, so there is no pool and no stream-ordered free.
template <typename T, bool kPinnedHost = false>
class Buffer {
 public:
  Buffer() = default;
  Buffer(const Buffer &) = delete;
  Buffer &operator=(const Buffer &) = delete;
  Buffer(Buffer &&o) noexcept : p_(std::exchange(o.p_, nullptr)), n_(std::exchange(o.n_, 0)) {}
  Buffer &operator=(Buffer &&o) noexcept {
    if (this != &o) {
      reset();
      p_ = std::exchange(o.p_, nullptr);
      n_ = std::exchange(o.n_, 0);
    }
    return *this;
  }
  ~Buffer() { reset(); }  // the status of the free is ignored, as in ials_trainer_destroy

  // n elements, contents undefined; whatever was held is freed first
  T *alloc(size_t n) {
    if (p_) CUDA_CHECK(reset());
    void *p = nullptr;
    if (kPinnedHost)
      CUDA_CHECK(cudaHostAlloc(&p, sizeof(T) * n, cudaHostAllocDefault));
    else
      CUDA_CHECK(cudaMalloc(&p, sizeof(T) * n));
    p_ = static_cast<T *>(p);
    n_ = n;
    return p_;
  }
  // grow-only: reallocates (the contents are not kept) when fewer than n elements are held
  T *ensure(size_t n) { return n > n_ ? alloc(n) : p_; }
  cudaError_t reset() {
    T *p = std::exchange(p_, nullptr);
    n_ = 0;
    if (!p) return cudaSuccess;
    return kPinnedHost ? cudaFreeHost(p) : cudaFree(p);
  }

  T *get() const { return p_; }
  size_t size() const { return n_; }

 private:
  T *p_ = nullptr;
  size_t n_ = 0;
};

template <typename T>
using DeviceBuffer = Buffer<T>;
template <typename T>
using PinnedBuffer = Buffer<T, true>;

// Declared after the temporary buffers of a call, these run before the buffers are freed, on the
// error path too: the work enqueued on them has finished (cudaFree is not relied on to wait for it).
struct StreamSyncOnExit {
  cudaStream_t s;
  ~StreamSyncOnExit() { cudaStreamSynchronize(s); }
};
struct DeviceSyncOnExit {
  ~DeviceSyncOnExit() { cudaDeviceSynchronize(); }
};

// Count of kernels launched by this library (bench.py reports it as gpu_launches).
extern int64_t g_kernel_launches;
inline void count_launch(int n = 1) { __atomic_fetch_add(&g_kernel_launches, (int64_t)n, __ATOMIC_RELAXED); }

__host__ __device__ inline int64_t round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }
__host__ __device__ inline int64_t ceil_div(int64_t x, int64_t m) { return (x + m - 1) / m; }

// Top-k sort key: (order-preserving bits of -score) << 32 | column id, so that ascending keys order
// by (-score, id) -- the reference's lexicographic pair comparison (evaluator.cpp:324-355)
__device__ __forceinline__ unsigned long long make_key(float s, uint32_t j) {
  s += 0.0f;  // -0.0 -> +0.0 so that equal scores compare equal, as floats do
  const uint32_t b = __float_as_uint(s);
  const uint32_t asc = (b & 0x80000000u) ? ~b : (b | 0x80000000u);
  return ((unsigned long long)(~asc) << 32) | j;
}
__device__ __forceinline__ float key_score(unsigned long long key) {
  const uint32_t asc = ~(uint32_t)(key >> 32);
  const uint32_t b = (asc & 0x80000000u) ? (asc & 0x7fffffffu) : ~asc;
  return __uint_as_float(b);
}

// Rows of a CSR whose neighbour lists are cut into jobs of <= job_len entries for the tensor-core
// Gram: the first n_heavy entries of the CSR's `order` (jobs of the h-th: [heavy_first_job[h],
// heavy_first_job[h + 1]))
struct JobPlan {
  int64_t n_heavy = 0, n_jobs = 0, nnz_heavy = 0;
  DeviceBuffer<int64_t> job_begin, job_end;  // [n_jobs]
  DeviceBuffer<int32_t> heavy_first_job;     // [n_heavy + 1]
};

// CSR in device memory.
struct DeviceCsr {
  int64_t n_rows = 0, n_cols = 0, nnz = 0;
  int64_t row_base = 0;  // global index of CSR row 0 (row shards; 0 for a full matrix)
  DeviceBuffer<int64_t> indptr;
  DeviceBuffer<int32_t> indices;
  DeviceBuffer<float> data;
  // rows sorted by descending degree (longest-processing-time-first schedule)
  DeviceBuffer<int32_t> order;
  int64_t max_degree = 0;
  JobPlan heavy;  // "heavy" rows (degree > threshold)
  bool has_negative = false;  // some stored value < 0: sqrt-weighted Gram not applicable
  int sorted_state = -1;      // column ids strictly ascending in every row? (-1: not checked yet)
};

// Arguments common to the per-row solvers (one half-epoch).
struct SolveArgs {
  float *target;          // [n_target x ld] rows being solved (in/out)
  const float *other;     // [n_other x ld]  gathered factor matrix
  const float *P;         // [ld x ld]       alpha0 * other^T other (symmetric)
  const int64_t *indptr;  // CSR of the target side
  const int32_t *indices;
  const float *data;
  const int32_t *order;   // schedule: order[s] = row solved s-th (may be null)
  int64_t n_rows;         // number of CSR rows
  int64_t n_sched;        // number of scheduled rows (entries of `order`, or n_rows)
  int64_t row_base;       // CSR row r solves target row row_base + r (row-sharded multi-GPU)
  int64_t n_other;
  int K;                  // true rank
  int ld;                 // padded row stride (multiple of 32)
  float alpha0, reg, nu, bias;
  int max_cg_steps;       // already resolved (0 -> K)
  int *err_flags;         // device, kNumErrFlags ints
  unsigned long long *work_counter;  // device, zeroed before launch
  // peer replicas of `target` (multi-GPU fused all-gather); n_peers may be 0
  int n_peers;
  float *peers[8];
  // cholesky_ll.cu only: row_jobs[slot .. slot + 1] = job range (absolute job ids) of the
  // slot-th scheduled row in the per-chunk workspace of Gram blocks
  const int32_t *row_jobs;
  // Warm starts that are still arriving from the host (ials_trainer_step_io): the rows
  // ready_base + [c << ready_shift, (c + 1) << ready_shift) of `target` are valid once
  // ready_flags[c] == ready_token.  nullptr: everything is resident.  (cg_rows.cu, dense_cg.cu)
  const int *ready_flags;
  int ready_token, ready_shift;
  int64_t ready_base;  // first factor row of chunk 0 (the shard's first row; 0 for a whole matrix)
  // Feature-aware iALS (Solver::step_cg with a prior, step_cholesky_with_prior,
  // IALSTrainer.hpp:170-271, 333-385): row u of `prior` ([n_target x ld], same rows as `target`)
  // enters the right-hand side as  b += reg_u * prior_u  and rows without interactions are solved
  // like the others.  nullptr: plain iALS.  (cg.cu, cholesky_tile.cu: the generic kernels)
  const float *prior;
};

// Spin until the chunk of `target` that holds factor row `gu` has landed (lane 0 / thread 0 of the
// caller, followed by the caller's own barrier).
__device__ __forceinline__ void wait_row_ready(const SolveArgs &a, int64_t gu) {
  const int *f = a.ready_flags + ((gu - a.ready_base) >> a.ready_shift);
  int v;
  for (;;) {
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
    if (v == a.ready_token) break;
    __nanosleep(256);
  }
}

// iALS++ subspace block [d0, d0 + S) of the factor (cholesky_tile.cu, SUB instantiation);
// pred[j] caches x_u . y_i for every stored entry j of the CSR being solved
struct SubspaceArgs {
  float *pred;
  int d0, S;
  // Explanations (cholesky_tile.cu, EXPLAIN instantiation; null in the others, whose parameter
  // offsets stay where they were because these follow): the scheduled slot s explains the pairs
  // [pair_ptr[s], pair_ptr[s + 1]) of its row, pair p against the row `targets[p]` of `other`;
  // score[p] = y_t . x_u, prior[p] = reg_u w_t . prior_u (optional), and the contribution
  // (bias + c_j) w_t . y_j of the row's j-th history entry goes to contrib[contrib_ptr[p] + j]
  // with its column id in contrib_idx, where w_t = A_u^-1 y_t.  Pair indices are slab-local.
  const int64_t *pair_ptr;
  const int32_t *targets;
  const int64_t *contrib_ptr;
  float *score, *prior, *contrib;
  int32_t *contrib_idx;
};

// Arguments of the tensor-core weighted Gram (wgram.cu).  Job j accumulates the entries
// [job_begin[j], job_end[j]) of (indices, weights) -- or, when indices == nullptr, the rows
// [job_begin[j], job_end[j]) of Y with unit weights -- and writes
//   W[j]      (128 x 128):  G_j = W_j + W_j^T = sum w y y^T
//   bpart[j]  (kWGramBParts x 128, optional): the producer warps' partial sums of (bias + w) y
struct WGramArgs {
  const float *Y;          // [n x ld] (may point into a wider row: Y + 128 with ld = 256)
  int ld;                  // row stride, >= 128
  const int32_t *indices;  // gathered row ids (nullptr: identity)
  const float *weights;    // (nullptr: 1)
  const int64_t *job_begin;
  const int64_t *job_end;
  int64_t n_jobs;
  float bias;
  float *W;
  float *bpart;
};

// Entries one operand list of the tensor-core Gram may hold: the producers of wgram.cu step int32
// offsets up to 32 entries past a job's end and read 31 past a stage's start.
constexpr int64_t kMaxGramEntries = (1ll << 31) - 64;

// ---- kernels / launchers (one .cu each) ----
void launch_wgram(const WGramArgs &a, cudaStream_t s);
void launch_wgram256(const WGramArgs &a, cudaStream_t s);  // whole Gram of 256-column rows: W [256][256] per job
void launch_wgram_reduce_sym(const float *W, int n_parts, float scale, float *out, cudaStream_t s);
constexpr int kWGramBParts = 16;  // producer warps of wgram.cu (one partial b each)
constexpr int kWGram256BParts = 8;  // producer warps of wgram256_kernel
// Workspace of the tensor-core K1 Gram: block jobs over contiguous rows + their partials.
struct GramWorkspace {
  int max_jobs = 0;
  DeviceBuffer<int64_t> job_begin, job_end;  // [max_jobs]
  DeviceBuffer<float> W;                     // [max_jobs x 128 x 128]
  void alloc(int jobs);
};
// P = alpha0 * Y[row_begin:row_end]^T Y[...] on tcgen05 (ld == 128 only)
void launch_gram_tc(const float *Y, int64_t row_begin, int64_t row_end, float alpha0,
                    const GramWorkspace &ws, float *P, cudaStream_t s);

void build_transpose(const DeviceCsr &X, DeviceCsr &Xt, cudaStream_t s);
void build_row_order(DeviceCsr &X, cudaStream_t s);
bool csr_has_negative(const DeviceCsr &X, cudaStream_t s);
// rows of X (in X.order) with more than `threshold` entries, cut into jobs of <= job_len entries
void build_heavy_plan(const DeviceCsr &X, int64_t threshold, int64_t job_len, JobPlan &plan, cudaStream_t s);
// Dense CG on explicitly formed normal equations (dense_cg.cu): heavy rows only.
struct DenseSolveArgs {
  SolveArgs base;                 // target / P / CSR / order / hyper-parameters / peers
  int64_t n_heavy;
  const int32_t *heavy_first_job; // [n_heavy + 1]
  const float *W;                 // [n_jobs x 128 x 128]  G_job = W + W^T
  const float *bpart;             // [n_jobs x kWGramBParts x 128]
  int job0;                       // ialspp_dense: W / bpart start at job `job0` (chunked workspace)
};
void launch_dense_cg(const DenseSolveArgs &a, cudaStream_t s);
// iALS++ as block Gauss-Seidel on the tensor-core Gram (ialspp_dense.cu): ld == 128, S <= 64
bool ialspp_dense_supported(const SolveArgs &a, int S);
void launch_ialspp_dense(const DenseSolveArgs &d, int S, int iters, cudaStream_t s);

void launch_gram(const float *Y, int64_t row_begin, int64_t row_end, int ld, float alpha0,
                 float *scratch /*ld*ld*/, float *P /*ld*ld*/, cudaStream_t s);

void launch_solve_cg_simple(const SolveArgs &a, cudaStream_t s);  // cg.cu: any row stride, warp per row
void launch_solve_cg_rows(const SolveArgs &a, cudaStream_t s);    // cg_rows.cu (ld == 128): two rows per warp
bool cholesky_tile_supported(const SolveArgs &a);                       // cholesky_tile.cu
void launch_solve_cholesky_tile(const SolveArgs &a, cudaStream_t s);  // register-tiled (default)
// iALS++ (Solver::step_ialspp, IALSTrainer.hpp:387-535), cholesky_tile.cu
void launch_ialspp_predict(const SolveArgs &a, float *pred, cudaStream_t s);
bool ialspp_block_supported(int S);
void launch_ialspp_block(const SolveArgs &a, float *pred, int d0, int S, cudaStream_t s);
// Explanations of scheduled rows (cholesky_tile.cu): `a` as for launch_solve_cholesky_tile (P, the
// history CSR, order = the rows to explain, prior), nothing written to a.target; `ex` as in SubspaceArgs.
// A row without history and without a prior is not solved: its scores and priors are 0.
void launch_explain_tile(const SolveArgs &a, const SubspaceArgs &ex, cudaStream_t s);

void launch_scores(const float *user_rows, int64_t n_rows, const float *item, int64_t n_items,
                   int ld, float *out, int64_t out_ld, cudaStream_t s);
void launch_mask_rows(float *scores, int64_t out_ld, const int64_t *indptr, const int32_t *indices,
                      const float *data, int64_t row0, int64_t n_rows, int64_t indptr_base,
                      cudaStream_t s);
// dst = -inf except at the allowed in-range columns (n_lists == 1: one list shared by all rows)
void launch_allow_rows(const float *src, float *dst, int64_t ld, const int64_t *indptr,
                       const int64_t *indices, int64_t n_lists, int64_t row0, int64_t n_rows,
                       int64_t n_items, cudaStream_t s);
void launch_topk_rows(const float *scores, int64_t out_ld, int64_t n_rows, int64_t n_items, int k,
                      int32_t *out_idx, float *out_score, int32_t *out_count, cudaStream_t s);

// candidates.cu: caller-given candidate lists, one CSR row of item ids per query row.  Row r of a
// slab reads list row0 + r (or list 0 for every row when shared_len >= 0) and keeps its scores in a
// scratch laid out in the same order, from position out(r).
struct CandSegments {
  const int64_t *indptr;
  const int32_t *indices;
  int64_t row0;        // list of slab row 0 (per-row lists)
  int64_t base;        // indptr[row0]: scratch position of slab row 0 (per-row lists)
  int64_t shared_len;  // >= 0: one list of this length shared by every row; -1: one list per row
  __device__ int64_t begin(int64_t r) const { return shared_len >= 0 ? 0 : indptr[row0 + r]; }
  __device__ int64_t end(int64_t r) const { return shared_len >= 0 ? shared_len : indptr[row0 + r + 1]; }
  __device__ int64_t out(int64_t r) const { return shared_len >= 0 ? r * shared_len : indptr[row0 + r] - base; }
};
// The items hidden from each query row (indptr == nullptr: none): CSR row row0 + r, or rowmap[r] + row0
// for users picked by index.  Entries whose data is 0 hide nothing (data may be null).  sorted: column
// ids strictly ascending in every row (binary search; otherwise the row is scanned).
struct CandMask {
  const int64_t *indptr = nullptr;
  const int32_t *indices = nullptr;
  const float *data = nullptr;
  int64_t row0 = 0;
  const int64_t *rowmap = nullptr;
  bool sorted = true;
};
// scores[out(r) + j] = queries[r] . item[list_r[j]] in FP32, -inf where the mask hides the item.  The work
// is cut into tasks of kCandChunk candidates of one row: row r owns tasks [tasks[r], tasks[r + 1]) (device,
// n_rows + 1 entries, ceil(length / kCandChunk) per row; tasks[0] need not be 0), n_tasks in all.
constexpr int kCandChunk = 256;
void launch_cand_scores(const float *queries, int64_t n_rows, int ld, const float *item, const CandSegments &seg,
                        const int64_t *tasks, int64_t n_tasks, const CandMask &mask, float *scores, cudaStream_t s);
// top-k of each row's segment of `scores` (candidates.cu), ordered by (-score, item id), -inf dropped.
// max_len, the longest list of the slab, picks the selection: a warp per row up to 256 candidates, a CTA
// per row above
void launch_topk_segments(const float *scores, const CandSegments &seg, int64_t n_rows, int64_t max_len, int k,
                          int32_t *out_idx, float *out_score, int32_t *out_count, cudaStream_t s);

// score_tc.cu: scores + seen mask + top-k fused on tcgen05 (ld a multiple of 32 in [32, 512],
// k <= 128; mask rows strictly ascending).  The dense score block (launch_scores_tc) takes
// ld <= 128 only: score_tc_supported(ld, 1).
bool score_tc_supported(int ld, int64_t k);
bool score_topk_tc_supported(int ld, int64_t k);
size_t score_tc_scratch_bytes(int64_t n_rows, int64_t n_items, int64_t k);
bool csr_rows_strictly_sorted(const int64_t *indptr, const int32_t *indices, int64_t n_rows,
                              cudaStream_t s);
// m_rowmap != nullptr: block row r is masked by CSR row m_row0 + m_rowmap[r] (users picked by index)
// a_n_lists >= 2: one allow-list per row (CSR, strictly ascending rows, row a_row0 + r);
// a_n_lists == 1: one list shared by every row, as a_bitmap (ceil(n_items / 32) words, bit = allowed)
void launch_score_topk_tc(const float *user_rows, int64_t n_rows, const float *item, int64_t n_items,
                          int ld, const int64_t *m_indptr, const int32_t *m_indices, const float *m_data,
                          int64_t m_row0, int k, void *scratch, int32_t *out_idx, float *out_score,
                          int32_t *out_count, cudaStream_t s, int a_n_lists = 0,
                          const int64_t *a_indptr = nullptr, const int32_t *a_indices = nullptr,
                          int64_t a_row0 = 0, const uint32_t *a_bitmap = nullptr,
                          const int64_t *m_rowmap = nullptr);
void launch_scores_tc(const float *user_rows, int64_t n_rows, const float *item, int64_t n_items, int ld,
                      float *out, int64_t out_ld, cudaStream_t s);

// prior_u / prior_i (optional): the side's regulariser is reg_u |x_u - prior_u|^2 (feature-aware)
void launch_loss(const float *user, const float *item, int64_t U, int64_t I, int K, int ld,
                 const DeviceCsr &X, const DeviceCsr &Xt, const float *Pu, const float *Pi,
                 float alpha0, float reg, float nu, float bias, const float *prior_u,
                 const float *prior_i, double *d_out, cudaStream_t s);
void launch_loss_add_sumsq(const float *v, int64_t n, float scale, double *d_out, cudaStream_t s);
// One rank's share of the sum of a row-sharded trainer: the rows X.row_base + [0, X.n_rows) of `user`
// and Xt.row_base + [0, Xt.n_rows) of `item` (full replicas); prior_u / prior_i hold those rows only;
// the Gram term is added when Pu != nullptr.  Zeroes *d_out first and leaves the sum un-halved.
void launch_loss_shard(const float *user, const float *item, int64_t U, int64_t I, int ld, const DeviceCsr &X,
                       const DeviceCsr &Xt, const float *Pu, const float *Pi, float alpha0, float reg, float nu,
                       float bias, const float *prior_u, const float *prior_i, double *d_out, cudaStream_t s);
void launch_loss_halve(double *d_out, cudaStream_t s);

// ---- feature-aware iALS (feature.cu; IALSTrainer.hpp:696-702, 1066-1209) ----
// A feature matrix on the device: dense row-major [n_rows x n_cols] or CSR.
struct FeatureDev {
  int64_t n_rows = 0, n_cols = 0, nnz = 0;
  const float *dense = nullptr;
  const int64_t *indptr = nullptr;
  const int32_t *indices = nullptr;
  const float *data = nullptr;
};
// out[r] = F[r] . W   (W [n_cols x ld], out [n_rows x ld]): feature_times_weight
void launch_feature_prior(const FeatureDev &F, const float *W, int ld, float *out, cudaStream_t s);
// rw[r] = reg * (alpha0 * n_other + nnz_r)^nu  (compute_reg per row of the CSR)
void launch_feature_row_weights(const int64_t *indptr, int64_t n_rows, int64_t n_other, float alpha0,
                                float reg, float nu, float *rw, cudaStream_t s);
// G [n_cols x n_cols] = F^T diag(rw) F + lambda I, then its Cholesky factor in place (lower);
// *fail (device int) is raised when a pivot is not positive
void launch_feature_gram_llt(const FeatureDev &F, const float *rw, float lambda, float *G, int *fail,
                             cudaStream_t s);
// R [n_cols x ld] = F^T diag(rw) X, then W = (L L^T)^-1 R in place (R becomes the weight);
// *fail is raised when the solution is not finite
void launch_feature_ridge_solve(const FeatureDev &F, const float *rw, const float *X, int ld,
                                const float *L, float *R, int *fail, cudaStream_t s);
// The two halves of each, for the row-sharded trainer, which all-reduces the F^T products in between:
// G = F^T diag(rw) F / R = F^T diag(rw) X over F's rows, and the steps that follow on the summed G / R
void launch_feature_gram(const FeatureDev &F, const float *rw, float *G, cudaStream_t s);
void launch_feature_llt(float *G, int64_t n, float lambda, int *fail, cudaStream_t s);
void launch_feature_rhs(const FeatureDev &F, const float *rw, const float *X, int ld, float *R, cudaStream_t s);
void launch_feature_solve(const float *L, int64_t n, float *R, int ld, int *fail, cudaStream_t s);

// ranking metrics of recommendation lists (metrics.cu).  rec [rows x k] holds lists of length k; each of
// the n_cut (<= kMaxMetricsCutoffs) device cutoffs (<= k) reads their prefix.  Per cutoff c:
// acc[c][5] += {hit, recall, ndcg, map, precision} sums, valid_user[c] / total_user[c] counts,
// item_cnt[c][n_items] += its histogram.  partial: metrics_partials(rows) x n_cut x 5 doubles of scratch.
// Deterministic: the float64 sums are added in a fixed order.
constexpr int kMaxMetricsCutoffs = 32;
int64_t metrics_partials(int64_t rows);
void launch_metrics_rows(const int32_t *rec, const int32_t *cnt, int64_t rows, int k, const int64_t *gt_indptr,
                         const int32_t *gt_indices, const double *discount, const double *cum_discount,
                         const int32_t *cutoffs, int n_cut, int recall_with_cutoff, int64_t n_items,
                         double *partial, double *acc, unsigned long long *valid_user,
                         unsigned long long *total_user, unsigned long long *item_cnt, cudaStream_t s);
// d_out[3] = {appeared_item, entropy, gini_index} of an item-count histogram (Metrics::as_dict without its
// sort); ws: grow-only workspace.  Synchronises the stream once (the count-of-counts table is sized by the
// largest count).
void diversity_of_histogram(const unsigned long long *hist, int64_t n_items, DeviceBuffer<unsigned char> &ws,
                            double *d_out, cudaStream_t s);
void launch_gather_rows(const float *src, int ld, const int64_t *rows, int64_t n_rows, float *dst,
                        cudaStream_t s);
void launch_pad_copy(const float *src, int64_t n_rows, int K, float *dst, int ld, cudaStream_t s);
// dst[r] = src[r] / |src[r]|, rows of norm 0 left at 0 (rows of ld floats, ld % 4 == 0)
void launch_normalize_rows(const float *src, int64_t n_rows, int ld, float *dst, cudaStream_t s);
// indptr[0 .. n] = 0 .. n, indices[0 .. n) = 0 .. n - 1: the mask CSR whose row i hides column i
void launch_self_mask(int64_t *indptr, int32_t *indices, int64_t n, cudaStream_t s);
void launch_unpad_copy(const float *src, int64_t n_rows, int K, int ld, float *dst, cudaStream_t s);
void launch_init_normal(float *dst, int64_t n_rows, int K, int ld, float stdev, uint64_t seed,
                        cudaStream_t s);

}  // namespace ials
