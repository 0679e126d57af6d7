// K2 conjugate-gradient row solve (replaces Solver::step_cg,
// /root/reference/cpp_source/als/IALSTrainer.hpp:170-271).
//
// Per row u with CSR neighbours (i, c), Y = other factors, P = alpha0 Y^T Y:
//   A = P + reg_u I + sum c y_i y_i^T,   b = sum (bias + c) y_i
//   x <- warm start;  r = b - A x;  p = r;  <= max_cg_steps CG iterations with
//   the reference's exits (||r||^2 <= 1e-20) and failure test (!(p.Ap > 0)).
// The b pass and the r-init pass are fused:  r = sum (bias + c - c (y.x)) y - P x - reg x
// so a row makes 1 + steps passes over its neighbour vectors instead of 2 + steps.
//
// This file holds the generic-K kernel: one warp per row, neighbour vectors re-read from
// global/L2 on every pass.  It works for every row stride (multiple of 32, <= 512) and serves
// the ranks above 128; K <= 128 (stride 128) runs cg_rows.cu / wgram.cu + dense_cg.cu.
#include "common.cuh"

namespace ials {
namespace {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <int NV>
__global__ void __launch_bounds__(128) cg_warp_kernel(SolveArgs a) {
  extern __shared__ float smem[];
  const int lane = threadIdx.x % kWarp;
  const int warp_in_block = threadIdx.x / kWarp;
  float *ps = smem + warp_in_block * a.ld;  // per-warp broadcast buffer for P*v products
  const int ld = a.ld;

  for (;;) {
    unsigned long long slot = 0;
    if (lane == 0) slot = atomicAdd(a.work_counter, 1ull);
    slot = __shfl_sync(0xffffffffu, slot, 0);
    if ((int64_t)slot >= a.n_sched) break;
    const int64_t u = a.order ? (int64_t)a.order[slot] : (int64_t)slot;  // CSR row
    const int64_t gu = a.row_base + u;                                   // factor row

    float *xrow = a.target + gu * ld;
    float x[NV], r[NV], p[NV], Ap[NV];
#pragma unroll
    for (int j = 0; j < NV; j++) x[j] = xrow[lane + 32 * j];
    const int64_t s = a.indptr[u], e = a.indptr[u + 1];
    const int64_t nnz = e - s;
    const float reg_u = a.reg * powf(a.alpha0 * (float)a.n_other + (float)nnz, a.nu);
    if (nnz == 0 && a.prior == nullptr) {  // :207-210 (with a prior the row is solved like the others)
#pragma unroll
      for (int j = 0; j < NV; j++) x[j] = 0.f;
    } else {
      // fused b / r-init pass; b starts from reg_u * prior_u in the feature-aware model (:212-216)
#pragma unroll
      for (int j = 0; j < NV; j++) r[j] = a.prior ? reg_u * a.prior[gu * ld + lane + 32 * j] : 0.f;
      for (int64_t jn = s; jn < e; jn++) {
        const float *v = a.other + (int64_t)a.indices[jn] * ld;
        const float c = a.data[jn];
        float vv[NV], d = 0.f;
#pragma unroll
        for (int j = 0; j < NV; j++) { vv[j] = v[lane + 32 * j]; d = fmaf(vv[j], x[j], d); }
        d = warp_sum(d);
        const float coef = (a.bias + c) - c * d;
#pragma unroll
        for (int j = 0; j < NV; j++) r[j] = fmaf(coef, vv[j], r[j]);
      }
      // r -= P x + reg_u x   (P symmetric: column access is coalesced)
      __syncwarp();
#pragma unroll
      for (int j = 0; j < NV; j++) ps[lane + 32 * j] = x[j];
      __syncwarp();
      {
        float acc[NV];
#pragma unroll
        for (int j = 0; j < NV; j++) acc[j] = 0.f;
        for (int k = 0; k < a.K; k++) {
          const float xk = ps[k];
          const float *Prow = a.P + (int64_t)k * ld;
#pragma unroll
          for (int j = 0; j < NV; j++) acc[j] = fmaf(Prow[lane + 32 * j], xk, acc[j]);
        }
#pragma unroll
        for (int j = 0; j < NV; j++) { r[j] -= acc[j]; r[j] = fmaf(-reg_u, x[j], r[j]); p[j] = r[j]; }
      }
      bool failed = false;
      for (int it = 0; it < a.max_cg_steps; it++) {
        float r2 = 0.f;
#pragma unroll
        for (int j = 0; j < NV; j++) r2 = fmaf(r[j], r[j], r2);
        r2 = warp_sum(r2);
        if (r2 <= 1e-20f) break;
        __syncwarp();
#pragma unroll
        for (int j = 0; j < NV; j++) ps[lane + 32 * j] = p[j];
        __syncwarp();
#pragma unroll
        for (int j = 0; j < NV; j++) Ap[j] = 0.f;
        for (int k = 0; k < a.K; k++) {
          const float pk = ps[k];
          const float *Prow = a.P + (int64_t)k * ld;
#pragma unroll
          for (int j = 0; j < NV; j++) Ap[j] = fmaf(Prow[lane + 32 * j], pk, Ap[j]);
        }
#pragma unroll
        for (int j = 0; j < NV; j++) Ap[j] = fmaf(reg_u, p[j], Ap[j]);
        for (int64_t jn = s; jn < e; jn++) {
          const float *v = a.other + (int64_t)a.indices[jn] * ld;
          const float c = a.data[jn];
          float vv[NV], d = 0.f;
#pragma unroll
          for (int j = 0; j < NV; j++) { vv[j] = v[lane + 32 * j]; d = fmaf(vv[j], p[j], d); }
          d = warp_sum(d);
          const float coef = c * d;
#pragma unroll
          for (int j = 0; j < NV; j++) Ap[j] = fmaf(coef, vv[j], Ap[j]);
        }
        float den = 0.f;
#pragma unroll
        for (int j = 0; j < NV; j++) den = fmaf(p[j], Ap[j], den);
        den = warp_sum(den);
        if (!(den > 0.f) || !isfinite(den)) { failed = true; break; }
        const float alpha = r2 / den;
        float r2n = 0.f;
#pragma unroll
        for (int j = 0; j < NV; j++) {
          x[j] = fmaf(alpha, p[j], x[j]);
          r[j] = fmaf(-alpha, Ap[j], r[j]);
          r2n = fmaf(r[j], r[j], r2n);
        }
        r2n = warp_sum(r2n);
        if (r2n <= 1e-20f) break;
        const float beta = r2n / r2;
#pragma unroll
        for (int j = 0; j < NV; j++) p[j] = fmaf(beta, p[j], r[j]);
      }
      if (failed) {
        if (lane == 0) atomicExch(&a.err_flags[kErrCgSingular], 1);
        continue;  // the reference throws before writing the row back
      }
    }
#pragma unroll
    for (int j = 0; j < NV; j++) xrow[lane + 32 * j] = x[j];
    for (int pi = 0; pi < a.n_peers; pi++) {
      float *prow = a.peers[pi] + gu * ld;
#pragma unroll
      for (int j = 0; j < NV; j++) prow[lane + 32 * j] = x[j];
    }
  }
}


template <int NV>
void launch_nv(const SolveArgs &a, cudaStream_t s) {
  const int threads = 128;
  const size_t smem = sizeof(float) * (threads / kWarp) * a.ld;
  const int64_t warps_needed = std::max<int64_t>(a.n_sched, 1);
  const unsigned grid = (unsigned)std::min<int64_t>(ceil_div(warps_needed, threads / kWarp),
                                                    (int64_t)kNumSMsB200 * 16);
  cg_warp_kernel<NV><<<grid, threads, smem, s>>>(a); count_launch();
  CUDA_CHECK(cudaGetLastError());
}

}  // namespace

void launch_solve_cg_simple(const SolveArgs &a, cudaStream_t s) {
  CUDA_CHECK(cudaMemsetAsync(a.work_counter, 0, sizeof(unsigned long long), s));
  switch (a.ld / 32) {
    case 1: launch_nv<1>(a, s); break;
    case 2: launch_nv<2>(a, s); break;
    case 3: launch_nv<3>(a, s); break;
    case 4: launch_nv<4>(a, s); break;
    case 5: launch_nv<5>(a, s); break;
    case 6: launch_nv<6>(a, s); break;
    case 7: launch_nv<7>(a, s); break;
    case 8: launch_nv<8>(a, s); break;
    case 9: launch_nv<9>(a, s); break;
    case 10: launch_nv<10>(a, s); break;
    case 11: launch_nv<11>(a, s); break;
    case 12: launch_nv<12>(a, s); break;
    case 13: launch_nv<13>(a, s); break;
    case 14: launch_nv<14>(a, s); break;
    case 15: launch_nv<15>(a, s); break;
    case 16: launch_nv<16>(a, s); break;
    default:  // new_trainer accepts K <= 512, so every stride it produces has a case above
      throw NotImplemented("CG solver: the row stride must be a multiple of 32 in [32, 512]");
  }
}

}  // namespace ials
