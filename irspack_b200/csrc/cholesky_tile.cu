// K3 Cholesky row solve, register-tiled (replaces Solver::step_cholesky + BatchedRankUpdater,
// /root/reference/cpp_source/als/IALSTrainer.hpp:273-331, 37-58).
//
// Per row:  A = P + sum c y y^T + reg_u I,  b = sum (bias + c) y,  A = U^T U,  U^T z = b,
// U x = z.  Empty rows are not special-cased (x = 0 falls out).
//
// ncu on the v0 kernel (cholesky.cu, profiles/r01l_prof_chol.md): 2.5 M warp instructions per
// row at K = 256, most of them the right-looking factorisation walking the packed triangle in
// shared memory one element per thread and step, plus the read-modify-write of every 8x8 tile
// after each rank-update stage (19 % of the shared-memory wavefronts are bank conflicts).
// Here the matrix never leaves the register file until it is final:
//   * thread t owns the 8x8 tile (ti, tj), tj >= ti, of A for the whole row: it is initialised
//     from P, takes the rank updates (neighbour vectors staged 32 at a time in shared memory,
//     rows padded so that the eight-float segments of a quarter warp hit distinct banks) and
//     the ridge on its diagonal;
//   * factorisation, BLOCKED by tile rows (8 pivots), two barriers per block instead of one
//     per pivot (r01l ncu: 52 % of the stall samples were per-pivot barrier waits):
//       phase 1  the tiles of tile row pb apply the 8 pivots' row operations to themselves with
//                the multipliers of the diagonal tile (64 floats in shared memory) and publish
//                their 8 final rows (unscaled) to a padded row block and to the packed factor;
//       phase 2  every tile below subtracts the rank-8 update  sum_li (a_r / a_ii) a_c  with
//                8 x (4 LDS.128 + 8 FMUL + 64 FFMA); the owner of the NEXT diagonal tile then
//                eliminates it on the spot and publishes its multipliers, so the serial 8-pivot
//                chain of a diagonal tile overlaps the other threads' phase 2;
//     the arithmetic per matrix element is the same FMA sequence as the pivot-by-pivot loop;
//     b rides along as an extra column, which is the forward substitution;
//   * the factor is kept UNSCALED (row i of U is published row / sqrt(a_ii)); one warp does the
//     backward substitution  x_i = (b_i - sum_{c>i} a_ic x_c) / a_ii  row by row with shuffle
//     reductions, no block barrier.
// One CTA per row, one thread per tile (528 tiles at K = 256 -> 544 threads, <= 120 registers).
//
// The SUB instantiation is the block solve of iALS++ (Solver::_step_dimrange,
// IALSTrainer.hpp:426-518): the system is the S x S block [d0, d0 + S) of the same matrix, the
// right-hand side is  P[d0:d0+S, :] x + reg x_S + sum (c (pred - 1) - bias) y_S,  the solution is
// SUBTRACTED from x_S and from the cached predictions of the row's entries (:499-508).
// ialspp_predict_kernel is Solver::_prediction (:387-424).
//
// The EXPLAIN instantiation splits scores into the contributions of the row's history (Hu, Koren and
// Volinsky, ICDM 2008, section 5): it forms and factors A_u exactly as MODE 0, keeps the factor in
// shared memory and, for each target t of the row, solves A_u w_t = y_t (one warp per target, the
// lane-register layout of the backward substitution below, up to kStage targets at a time in V).
// The history rows are then read once per group of targets:  score(u, t) = y_t . x_u
// = sum_j (bias + c_j) w_t . y_j + reg_u w_t . prior_u.
#include "common.cuh"

namespace ials {
namespace {

constexpr int kMaxThreads = 544;
constexpr int kStage = 32;  // neighbours staged per rank-update step

__device__ __host__ __forceinline__ int pad8(int c) { return c + ((c >> 3) << 2); }  // 8 floats -> 12
__device__ __forceinline__ int packed_row(int i, int kd) { return i * kd - (i * (i - 1)) / 2; }  // (i, i)

// The tile lives in registers as 8 x 4 pairs so that the two hot loops (rank update, trailing
// update) run on packed FP32 (sm_100 fma.rn.f32x2 -> FFMA2: two fused multiply-adds per issue
// slot; the kernel is bound by instruction issue, ncu r01l: fma pipe 18 %, issue 33 % at 17 warps).
// EL(i, j) names one element; i and j are compile-time constants wherever it is used.
#define EL(i, j) (((j) & 1) ? acc[i][(j) >> 1].y : acc[i][(j) >> 1].x)
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) {
  float2 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;"
      : "=l"(*reinterpret_cast<unsigned long long *>(&d))
      : "l"(*reinterpret_cast<unsigned long long *>(&a)), "l"(*reinterpret_cast<unsigned long long *>(&b)),
        "l"(*reinterpret_cast<unsigned long long *>(&c)));
  return d;
}

struct TileSmem {
  float *U;      // packed upper triangle, unscaled pivot rows: row i at packed_row(i), kd - i floats
  float *V;      // [kStage][pad8(kd)] staged neighbour vectors
  float *prow;   // [8][pad8(kd)] the 8 pivot rows of the current block (unscaled)
  float *mult;   // [64] multipliers a_ir / a_ii of the current diagonal tile (i < r within the tile)
  float *b;      // [kd] right-hand side / forward-substituted
  float *dinv;   // [kd] 1 / a_ii (the pivot before the square root)
  float *x;      // [kd] solution
  float *cw;     // [kStage] confidences of the staged neighbours (weights of the rank update)
  float *cwb;    // [kStage] their weights in the right-hand side
};
__host__ __device__ inline size_t tile_smem_floats(int kd) {
  const size_t packed = ((size_t)kd * (kd + 1) / 2 + 3) & ~(size_t)3;
  return packed + (size_t)kStage * pad8(kd) + 8 * (size_t)pad8(kd) + 64 + 3 * (size_t)kd + 2 * kStage;
}

// MODE 0: Solver::step_cholesky; 1 (SUB): the iALS++ block; 2 (EXPLAIN): explanations, see the
// header.  (256-column factors take the tensor-core Gram + cholesky_ll.cu instead; this kernel stays
// their fallback for rows with negative stored values and for IALS_CHOL=simt.)
template <int MODE>
__global__ void __launch_bounds__(kMaxThreads, 1) cholesky_tile_kernel(SolveArgs a, SubspaceArgs sub) {
  constexpr bool SUB = MODE == 1;
  constexpr bool EXPLAIN = MODE == 2;
  extern __shared__ __align__(16) float smem[];
  const int ld = a.ld;
  const int K = SUB ? sub.S : a.K;   // order of the system
  const int d0 = SUB ? sub.d0 : 0;   // first factor column of the system
  const int kd = SUB ? ((K + 7) & ~7) : min(ld, (K + 7) & ~7);  // columns that can be non-zero
  const int nt = kd / 8;
  const int n_tiles = nt * (nt + 1) / 2;
  const int kp = pad8(kd);
  TileSmem sm;
  sm.U = smem;
  sm.V = sm.U + (((size_t)kd * (kd + 1) / 2 + 3) & ~(size_t)3);
  sm.prow = sm.V + (size_t)kStage * kp;
  sm.mult = sm.prow + 8 * kp;
  sm.b = sm.mult + 64;
  sm.dinv = sm.b + kd;
  sm.x = sm.dinv + kd;
  sm.cw = sm.x + kd;
  sm.cwb = sm.cw + kStage;
  __shared__ long long s_slot;
  __shared__ int s_fail;
  const int tid = threadIdx.x, lane = tid % kWarp, warp = tid / kWarp;
  const int n_threads = blockDim.x, n_warps = n_threads / kWarp;

  // this thread's tile: row-major over the upper triangle of the nt x nt tile grid
  const bool has_tile = tid < n_tiles;
  int ti = 0, tj = 0;
  if (has_tile) {
    int rem = tid;
    while (rem >= nt - ti) {
      rem -= nt - ti;
      ti++;
    }
    tj = ti + rem;
  }
  const int i0 = ti * 8, j0 = tj * 8;

  for (;;) {
    __syncthreads();
    if (tid == 0) {
      s_slot = (long long)atomicAdd(a.work_counter, 1ull);
      s_fail = 0;
    }
    __syncthreads();
    const int64_t slot = s_slot;
    if (slot >= a.n_sched) break;
    const int64_t u = a.order ? (int64_t)a.order[slot] : slot;  // CSR row
    const int64_t gu = a.row_base + u;                          // factor row

    const int64_t s = a.indptr[u], e = a.indptr[u + 1];
    const int64_t nnz = e - s;
    const float reg_u = a.reg * powf(a.alpha0 * (float)a.n_other + (float)nnz, a.nu);  // :309-310
    const float *xrow = a.target + gu * ld;
    if (EXPLAIN && nnz == 0 && a.prior == nullptr) {  // x = 0 (cg_warp_kernel's), nothing to solve
      for (int64_t p = sub.pair_ptr[slot] + tid; p < sub.pair_ptr[slot + 1]; p += n_threads) {
        sub.score[p] = 0.f;
        if (sub.prior) sub.prior[p] = 0.f;
      }
      continue;
    }

    // acc <- P tile, b <- 0                                        (:296-299)
    float2 acc[8][4];
    if (has_tile) {
      if (!SUB) {
#pragma unroll
        for (int i = 0; i < 8; i++) {
          const float4 p0 = *reinterpret_cast<const float4 *>(a.P + (size_t)(i0 + i) * ld + j0);
          const float4 p1 = *reinterpret_cast<const float4 *>(a.P + (size_t)(i0 + i) * ld + j0 + 4);
          acc[i][0] = make_float2(p0.x, p0.y); acc[i][1] = make_float2(p0.z, p0.w);
          acc[i][2] = make_float2(p1.x, p1.y); acc[i][3] = make_float2(p1.z, p1.w);
        }
      } else {  // P_quadratic (:445-446): d0 need not be a multiple of four, scalar loads
#pragma unroll
        for (int i = 0; i < 8; i++)
#pragma unroll
          for (int j = 0; j < 8; j++)
            EL(i, j) = (i0 + i < K && j0 + j < K) ? a.P[(size_t)(d0 + i0 + i) * ld + d0 + j0 + j] : 0.f;
      }
    }
    if (!SUB) {  // step_cholesky_with_prior (:362): b starts from reg_u * prior_u
      for (int k = tid; k < kd; k += n_threads) sm.b[k] = (a.prior && k < K) ? reg_u * a.prior[gu * ld + k] : 0.f;
    } else {  // b <- P[d0:d0+S, :] x + reg x_S (:474-478), one warp per entry
      for (int k = warp; k < kd; k += n_warps) {
        float part = 0.f;
        if (k < K) {
          const float *Prow = a.P + (size_t)(d0 + k) * ld;
          for (int c = lane; c < ld; c += kWarp) part = fmaf(Prow[c], xrow[c], part);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
        if (lane == 0) sm.b[k] = k < K ? fmaf(reg_u, xrow[d0 + k], part) : 0.f;
      }
    }

    for (int64_t base = s; base < e; base += kStage) {  // rank updates (:301-308)
      const int m = (int)min((int64_t)kStage, e - base);
      __syncthreads();  // the previous stage is consumed (and b is zeroed)
      for (int t = warp; t < m; t += n_warps) {
        const float *v = a.other + (int64_t)a.indices[base + t] * ld + d0;
        if (!SUB) {
          for (int k = lane * 4; k < kd; k += kWarp * 4)
            *reinterpret_cast<float4 *>(&sm.V[t * kp + pad8(k)]) = *reinterpret_cast<const float4 *>(v + k);
        } else {  // columns [d0, d0 + S) only; the padding up to kd must be zero
          for (int k = lane; k < kd; k += kWarp) sm.V[t * kp + pad8(k)] = k < K ? v[k] : 0.f;
        }
        if (lane == 0) {
          const float c = a.data[base + t];
          sm.cw[t] = c;
          // (:301-307) b += (bias + c) y;  iALS++ (:486-490) b += (c (pred - 1) - bias) y_S
          sm.cwb[t] = SUB ? c * (sub.pred[base + t] - 1.f) - a.bias : a.bias + c;
        }
      }
      __syncthreads();
      for (int k = tid; k < kd; k += n_threads) {
        float bk = sm.b[k];
        const int kk = pad8(k);
        for (int t = 0; t < m; t++) bk = fmaf(sm.cwb[t], sm.V[t * kp + kk], bk);
        sm.b[k] = bk;
      }
      if (has_tile) {
        const float *va = sm.V + pad8(i0), *vb = sm.V + pad8(j0);
        for (int q = 0; q < m; q++) {
          const float c = sm.cw[q];
          const float4 a0 = *reinterpret_cast<const float4 *>(va + q * kp);
          const float4 a1 = *reinterpret_cast<const float4 *>(va + q * kp + 4);
          const float4 b0 = *reinterpret_cast<const float4 *>(vb + q * kp);
          const float4 b1 = *reinterpret_cast<const float4 *>(vb + q * kp + 4);
          const float av[8] = {c * a0.x, c * a0.y, c * a0.z, c * a0.w, c * a1.x, c * a1.y, c * a1.z, c * a1.w};
          const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
          for (int i = 0; i < 8; i++)
#pragma unroll
            for (int j = 0; j < 4; j++)
              acc[i][j] = fma2(make_float2(av[i], av[i]), make_float2(bv[2 * j], bv[2 * j + 1]), acc[i][j]);
        }
      }
    }
    if (has_tile && ti == tj) {  // :312-314
#pragma unroll
      for (int i = 0; i < 8; i++)
        if (i0 + i < K) EL(i, i) += reg_u;
    }
    __syncthreads();  // b is complete

    // right-looking Cholesky of the leading K x K block, b as an extra column    (:316-319),
    // blocked by tile rows (see the header)
    bool failed = false;
    // eliminate a diagonal tile in registers: multipliers -> sm.mult, 1 / pivot -> sm.dinv
    auto eliminate_diagonal = [&](int pb) {
      const int nl = min(8, K - 8 * pb);
#pragma unroll
      for (int li = 0; li < 8; li++) {
        if (li < nl) {
          const float d2 = EL(li, li);
          if (!(d2 > 0.f)) s_fail = 1;
          const float inv2 = 1.0f / d2;
          sm.dinv[8 * pb + li] = inv2;
#pragma unroll
          for (int r = 0; r < 8; r++) {
            if (r > li) {
              const float m = EL(li, r) * inv2;
              sm.mult[li * 8 + r] = m;
#pragma unroll
              for (int j = 0; j < 4; j++) acc[r][j] = fma2(make_float2(-m, -m), acc[li][j], acc[r][j]);
            }
          }
        }
      }
    };
    if (has_tile && ti == 0 && tj == 0) eliminate_diagonal(0);
    __syncthreads();
    const int n_blocks = (K + 7) / 8;
    for (int pb = 0; pb < n_blocks; pb++) {
      if (s_fail) {  // uniform: written before the barrier every thread just passed
        failed = true;
        break;
      }
      const int nl = min(8, K - 8 * pb);
      // ---- phase 1: tile row pb finishes its 8 rows and publishes them ----
      if (has_tile && ti == pb) {
        if (tj != pb) {
#pragma unroll
          for (int li = 0; li < 8; li++) {
            if (li < nl) {
#pragma unroll
              for (int r = 0; r < 8; r++) {
                if (r > li) {
                  const float m = sm.mult[li * 8 + r];
#pragma unroll
                  for (int j = 0; j < 4; j++) acc[r][j] = fma2(make_float2(-m, -m), acc[li][j], acc[r][j]);
                }
              }
            }
          }
        } else {  // the diagonal tile's owner: forward substitution inside the block
#pragma unroll
          for (int li = 0; li < 8; li++) {
            if (li < nl) {  // b_k -= a_ik (b_i / a_ii), the pivot loop's operation order
              const float bi = sm.b[8 * pb + li] * sm.dinv[8 * pb + li];
#pragma unroll
              for (int r = 0; r < 8; r++)
                if (r > li) sm.b[8 * pb + r] = fmaf(-EL(li, r), bi, sm.b[8 * pb + r]);
            }
          }
        }
#pragma unroll
        for (int li = 0; li < 8; li++) {
          if (li < nl) {
            const int i = 8 * pb + li;
            float *Ui = sm.U + packed_row(i, kd) - i;  // Ui[c] = (i, c)
            float *pr = sm.prow + li * kp + pad8(j0);
#pragma unroll
            for (int j = 0; j < 8; j++) {
              pr[j] = EL(li, j);
              if (j0 + j >= i) Ui[j0 + j] = EL(li, j);
            }
          }
        }
      }
      __syncthreads();
      // ---- phase 2: rank-nl update of everything below; b rides along ----
      for (int k = 8 * pb + 8 + tid; k < kd; k += n_threads) {
        float bk = sm.b[k];
        const int kk = pad8(k);
#pragma unroll
        for (int li = 0; li < 8; li++)
          if (li < nl) bk = fmaf(-sm.prow[li * kp + kk], sm.b[8 * pb + li] * sm.dinv[8 * pb + li], bk);
        sm.b[k] = bk;
      }
      if (has_tile && ti > pb) {
#pragma unroll
        for (int li = 0; li < 8; li++) {
          if (li < nl) {
            const float inv2 = sm.dinv[8 * pb + li];
            const float *pr = sm.prow + li * kp;
            const float4 r0 = *reinterpret_cast<const float4 *>(pr + pad8(i0));
            const float4 r1 = *reinterpret_cast<const float4 *>(pr + pad8(i0) + 4);
            const float4 c0 = *reinterpret_cast<const float4 *>(pr + pad8(j0));
            const float4 c1 = *reinterpret_cast<const float4 *>(pr + pad8(j0) + 4);
            const float ur[8] = {r0.x * inv2, r0.y * inv2, r0.z * inv2, r0.w * inv2,
                                 r1.x * inv2, r1.y * inv2, r1.z * inv2, r1.w * inv2};
            const float uc[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
#pragma unroll
            for (int r = 0; r < 8; r++)
#pragma unroll
              for (int j = 0; j < 4; j++)
                acc[r][j] = fma2(make_float2(-ur[r], -ur[r]), make_float2(uc[2 * j], uc[2 * j + 1]), acc[r][j]);
          }
        }
        // look-ahead: the next diagonal tile is final now; its owner eliminates it while the
        // other threads are still in their phase 2
        if (ti == pb + 1 && tj == pb + 1 && pb + 1 < n_blocks) eliminate_diagonal(pb + 1);
      }
      __syncthreads();
    }
    __syncthreads();
    if (failed) {
      if (tid == 0) atomicExch(&a.err_flags[kErrCholDecomp], 1);
      continue;
    }

    // backward substitution by one warp:  x_i = (b_i - sum_{c > i} a_ic x_c) / a_ii.
    // x stays in registers (lane l holds x_l, x_{l+32}, ...): per pivot one round of
    // independent LDS, a butterfly sum that leaves x_i in every lane, no barrier
    // (profiles/r01l_tile_prof_chol_tile.md: the shared-memory version of this loop held the
    // other 16 warps at the barrier for 31 % of the kernel).
    if (warp == 0) {
      constexpr int NX = 8;  // kd <= 256 (cholesky_tile_supported)
      float xr[NX];
#pragma unroll
      for (int j = 0; j < NX; j++) xr[j] = 0.f;
      for (int i = K - 1; i >= 0; i--) {
        const float *Ui = sm.U + packed_row(i, kd) - i;
        const float bi = sm.b[i], di = sm.dinv[i];
        float part = 0.f;
#pragma unroll
        for (int j = 0; j < NX; j++) {
          const int c = lane + 32 * j;
          if (c > i && c < K) part = fmaf(Ui[c], xr[j], part);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
        const float xi = (bi - part) * di;
#pragma unroll
        for (int j = 0; j < NX; j++)  // selects, so that xr stays in registers
          xr[j] = (j == (i >> 5) && lane == (i & 31)) ? xi : xr[j];
      }
#pragma unroll
      for (int j = 0; j < NX; j++) {
        const int c = lane + 32 * j;
        if (c < K) sm.x[c] = xr[j];
      }
    }
    __syncthreads();
    bool finite = true;
    for (int k = tid; k < K; k += n_threads) finite = finite && isfinite(sm.x[k]);
    if (!finite) s_fail = 1;
    __syncthreads();
    if (s_fail) {  // :320-323
      if (tid == 0) atomicExch(&a.err_flags[kErrCholSolve], 1);
      continue;
    }
    if (MODE == 0) {
      for (int k = tid; k < ld; k += n_threads) {
        const float v = k < K ? sm.x[k] : 0.f;
        a.target[gu * ld + k] = v;
        for (int pi = 0; pi < a.n_peers; pi++) a.peers[pi][gu * ld + k] = v;
      }
    } else if (SUB) {  // x_S -= delta, pred -= delta . y_S  (:499-508)
      for (int k = tid; k < K; k += n_threads) {
        const float v = xrow[d0 + k] - sm.x[k];
        a.target[gu * ld + d0 + k] = v;
        for (int pi = 0; pi < a.n_peers; pi++) a.peers[pi][gu * ld + d0 + k] = v;
      }
      for (int64_t j = s + warp; j < e; j += n_warps) {
        const float *v = a.other + (int64_t)a.indices[j] * ld + d0;
        float part = 0.f;
        for (int k = lane; k < K; k += kWarp) part = fmaf(sm.x[k], v[k], part);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
        if (lane == 0) sub.pred[j] -= part;
      }
    } else {  // EXPLAIN
      constexpr int NX = 8;
      const unsigned full = 0xffffffffu;
      const float *prior_u = a.prior ? a.prior + gu * ld : nullptr;
      const int64_t p0 = sub.pair_ptr[slot], p1 = sub.pair_ptr[slot + 1];
      for (int64_t g0 = p0; g0 < p1; g0 += kStage) {
        const int m = (int)min((int64_t)kStage, p1 - g0);
        __syncthreads();  // V is free: the rank updates (or the previous group) are done with it
        // w_t = A^-1 y_t by warp, t < m:  U^T D^-1 z = y  (z_c -= a_ic z_i / a_ii, the forward
        // substitution of the factorisation), then U w = z as the backward substitution above
        for (int t = warp; t < m; t += n_warps) {
          const float *y = a.other + (int64_t)sub.targets[g0 + t] * ld;
          float zr[NX];  // z, then w from the back: w_c for c > i, z_c for c <= i at pivot i
#pragma unroll
          for (int j = 0; j < NX; j++) {
            const int c = lane + 32 * j;
            zr[j] = c < K ? y[c] : 0.f;
          }
#pragma unroll
          for (int jb = 0; jb < NX; jb++) {
            for (int il = 0; il < kWarp && 32 * jb + il < K; il++) {
              const int i = 32 * jb + il;
              const float zi = __shfl_sync(full, zr[jb], il) * sm.dinv[i];
              const float *Ui = sm.U + packed_row(i, kd) - i;
#pragma unroll
              for (int j = jb; j < NX; j++) {
                const int c = lane + 32 * j;
                if (c > i && c < K) zr[j] = fmaf(-Ui[c], zi, zr[j]);
              }
            }
          }
#pragma unroll
          for (int jb = NX - 1; jb >= 0; jb--) {
            for (int il = min(kWarp, K - 32 * jb) - 1; il >= 0; il--) {
              const int i = 32 * jb + il;
              const float *Ui = sm.U + packed_row(i, kd) - i;
              float part = 0.f;
#pragma unroll
              for (int j = jb; j < NX; j++) {
                const int c = lane + 32 * j;
                if (c > i && c < K) part = fmaf(Ui[c], zr[j], part);
              }
#pragma unroll
              for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(full, part, o);
              const float wi = (__shfl_sync(full, zr[jb], il) - part) * sm.dinv[i];
              zr[jb] = lane == il ? wi : zr[jb];
            }
          }
#pragma unroll
          for (int j = 0; j < NX; j++) {  // V[c][t] (kStage x kd floats of the kStage x kp)
            const int c = lane + 32 * j;
            if (c < kd) sm.V[c * kStage + t] = zr[j];
          }
        }
        __syncthreads();
        // one warp per history entry j, lane t forms w_t . y_j: y_j is read once per group of targets
        // (the same address in every lane), the columns of V without bank conflicts
        for (int64_t j = s + warp; j < e; j += n_warps) {
          const int32_t col = a.indices[j];
          const float4 *y = reinterpret_cast<const float4 *>(a.other + (int64_t)col * ld);
          const float *v = sm.V + lane;
          float d0 = 0.f, d1 = 0.f, d2 = 0.f, d3 = 0.f;
          for (int c = 0; c < kd; c += 4, v += 4 * kStage) {  // w_t is 0 in the columns [K, kd)
            const float4 yc = __ldg(y + c / 4);
            d0 = fmaf(yc.x, v[0], d0);
            d1 = fmaf(yc.y, v[kStage], d1);
            d2 = fmaf(yc.z, v[2 * kStage], d2);
            d3 = fmaf(yc.w, v[3 * kStage], d3);
          }
          if (lane < m) {
            const int64_t o = sub.contrib_ptr[g0 + lane] + (j - s);
            sub.contrib[o] = (a.bias + a.data[j]) * ((d0 + d1) + (d2 + d3));
            sub.contrib_idx[o] = col;
          }
        }
        // score_t = y_t . x (computed apart from the contributions), prior_t = reg_u w_t . prior_u
        for (int t = warp; t < m; t += n_warps) {
          const float *y = a.other + (int64_t)sub.targets[g0 + t] * ld;
          float sc = 0.f, pr = 0.f;
          for (int c = lane; c < K; c += kWarp) {
            sc = fmaf(y[c], sm.x[c], sc);
            if (prior_u) pr = fmaf(sm.V[c * kStage + t], prior_u[c], pr);
          }
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) {
            sc += __shfl_xor_sync(full, sc, o);
            pr += __shfl_xor_sync(full, pr, o);
          }
          if (lane == 0) {
            sub.score[g0 + t] = sc;
            if (sub.prior) sub.prior[g0 + t] = prior_u ? reg_u * pr : 0.f;
          }
        }
      }
    }
  }
}

// Solver::_prediction (IALSTrainer.hpp:387-424): pred_j = x_u . y_i for every stored (u, i).
// One CTA per row off a dynamic cursor in schedule order, warps stride over the row's entries.
constexpr int kPredictThreads = 256;
__global__ void __launch_bounds__(kPredictThreads) ialspp_predict_kernel(SolveArgs a, float *pred) {
  __shared__ long long s_slot;
  const int lane = threadIdx.x % kWarp, warp = threadIdx.x / kWarp;
  constexpr int n_warps = kPredictThreads / kWarp;
  for (;;) {
    __syncthreads();
    if (threadIdx.x == 0) s_slot = (long long)atomicAdd(a.work_counter, 1ull);
    __syncthreads();
    const int64_t slot = s_slot;
    if (slot >= a.n_sched) break;
    const int64_t u = a.order ? (int64_t)a.order[slot] : slot;
    const float *x = a.target + (a.row_base + u) * a.ld;
    for (int64_t j = a.indptr[u] + warp; j < a.indptr[u + 1]; j += n_warps) {
      const float *y = a.other + (int64_t)a.indices[j] * a.ld;
      float part = 0.f;
      for (int k = lane; k < a.ld; k += kWarp) part = fmaf(x[k], y[k], part);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
      if (lane == 0) pred[j] = part;
    }
  }
}

}  // namespace

namespace {
int tile_system_kd(const SolveArgs &a, int S) {  // S < 0: the whole K x K system
  return S < 0 ? std::min(a.ld, (a.K + 7) & ~7) : (S + 7) & ~7;
}
bool tile_kd_supported(int kd) {
  const int nt = kd / 8;
  return nt >= 1 && nt * (nt + 1) / 2 <= kMaxThreads &&
         tile_smem_floats(kd) * sizeof(float) + 64 <= 227 * 1024;
}
template <int MODE>
void launch_tile(const SolveArgs &a, const SubspaceArgs &sub, int kd, cudaStream_t s) {
  const int nt = kd / 8;
  const int n_tiles = nt * (nt + 1) / 2;
  const size_t smem = tile_smem_floats(kd) * sizeof(float);
  const int threads = (int)round_up(std::max(std::max(n_tiles, kd), 64), 32);
  CUDA_CHECK(cudaMemsetAsync(a.work_counter, 0, sizeof(unsigned long long), s));
  CUDA_CHECK(cudaFuncSetAttribute(cholesky_tile_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)smem));
  int dev = 0, sms = kNumSMsB200;
  CUDA_CHECK(cudaGetDevice(&dev));
  CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  // resident CTAs per SM: shared memory, 120 registers per thread, 2048 threads
  const int by_smem = (int)((227 * 1024) / (smem + 1024));
  const int by_regs = 65536 / (threads * 120);
  const int per_sm = std::max(1, std::min(std::min(by_smem, by_regs), std::min(2048 / threads, 8)));
  const unsigned grid =
      (unsigned)std::min<int64_t>(std::max<int64_t>(a.n_sched, 1), (int64_t)sms * per_sm);
  cholesky_tile_kernel<MODE><<<grid, threads, smem, s>>>(a, sub);
  count_launch();
  CUDA_CHECK(cudaGetLastError());
}
}  // namespace

bool cholesky_tile_supported(const SolveArgs &a) { return tile_kd_supported(tile_system_kd(a, -1)); }

void launch_solve_cholesky_tile(const SolveArgs &a, cudaStream_t s) {
  if (!cholesky_tile_supported(a)) throw NotImplemented("Cholesky solver: n_components > 256 not supported");
  launch_tile<0>(a, SubspaceArgs{nullptr, 0, 0}, tile_system_kd(a, -1), s);
}

// iALS++: predictions of every stored entry, then one subspace block for every row
void launch_ialspp_predict(const SolveArgs &a, float *pred, cudaStream_t s) {
  if (a.n_sched <= 0) return;
  CUDA_CHECK(cudaMemsetAsync(a.work_counter, 0, sizeof(unsigned long long), s));
  int dev = 0, sms = kNumSMsB200;
  CUDA_CHECK(cudaGetDevice(&dev));
  CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const unsigned grid = (unsigned)std::min<int64_t>(a.n_sched, (int64_t)sms * 8);
  ialspp_predict_kernel<<<grid, kPredictThreads, 0, s>>>(a, pred);
  count_launch();
  CUDA_CHECK(cudaGetLastError());
}

bool ialspp_block_supported(int S) { return S >= 1 && tile_kd_supported((S + 7) & ~7); }

void launch_explain_tile(const SolveArgs &a, const SubspaceArgs &ex, cudaStream_t s) {
  if (a.n_sched <= 0) return;
  if (!cholesky_tile_supported(a)) throw NotImplemented("explanations: n_components > 256 not supported");
  launch_tile<2>(a, ex, tile_system_kd(a, -1), s);
}

void launch_ialspp_block(const SolveArgs &a, float *pred, int d0, int S, cudaStream_t s) {
  if (a.n_sched <= 0) return;
  if (!ialspp_block_supported(S)) throw NotImplemented("iALS++: ialspp_subspace_dimension > 256 not supported");
  if (d0 < 0 || d0 + S > a.K) throw InvalidArgument("iALS++: subspace block outside the factor");
  launch_tile<1>(a, SubspaceArgs{pred, d0, S}, tile_system_kd(a, S), s);
}

}  // namespace ials
