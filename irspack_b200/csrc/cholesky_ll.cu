// K3 Cholesky row solve for 256-column factors, after the tensor-core Gram (replaces
// Solver::step_cholesky, /root/reference/cpp_source/als/IALSTrainer.hpp:273-331, for the rows whose
// rank updates -- BatchedRankUpdater, :37-58 -- were done by wgram.cu; solve.cu solve_cholesky_tensor).
//
// Per row:  A = P + G + reg_u I  (G = sum c y y^T from the Gram workspace),  A = U^T U,
// U^T z = b,  U x = z.
//
// profiles/r02h: the register-tiled kernel (cholesky_tile.cu, one CTA of 544 threads = one row per
// SM, the matrix in registers, the factor in 131 KB of shared memory) spent 410 k cycles per row
// where the FMA work needs 11 k: one row per SM means every serial chain -- the 8-pivot diagonal
// eliminations, the 64 block barriers, the one-warp backward substitution -- is exposed.  Here the
// factor lives in a per-CTA scratch in GLOBAL memory (L2-resident: 152 KB per CTA), a CTA is 128
// threads and holds only ONE BLOCK ROW (32 x 256) of the matrix in registers, so four rows are in
// flight per SM and the chains of one row hide behind the FMAs of the others:
//   * blocked LEFT-looking factorisation, 8 block rows of 32: block row p starts from zero,
//     accumulates  S = sum_{k < 32 p} U(k, rows)^T U(k, cols)  from the finished block rows, which
//     are streamed from the scratch through shared memory (cp.async, 16 pivots per stage, double
//     buffered: 4 LDS.128 per 32 packed FFMA2), then takes  A - S  (A read once from the Gram
//     workspace + P, L2-prefetched while the stages run);
//   * during the accumulation thread (tr, tc) = (t & 3, t >> 2) owns the 8 x 8 tile (tr, tc) of
//     the block row: 4 tile rows x 32 tile columns; the tile columns left of the diagonal block
//     do not exist, so the live threads of the later block rows fill whole warps and the idle
//     warps cost nothing; the right-hand side is a 33rd tile column (column 0 = b: the forward
//     substitution is part of the factorisation) owned by four threads of warp 0 whose own tiles
//     lie below the diagonal;
//   * the block row itself: the tiles go to shared memory, warp 0 factors the 32 x 32 diagonal
//     block (lane = column, the scaled pivot row broadcast through shared memory), then every
//     thread owns two whole COLUMNS of the 32 x (W - 32 + 1) panel and solves them against the
//     triangle (packed FFMA2, the triangle broadcast from shared memory): 4 barriers per block
//     row, no divergence (the first version, r02j, did 4 steps of 8 pivots on the tiles: 48 % of
//     its stall samples were block barriers and a third of its instructions ran in half-empty
//     warps);
//   * backward substitution block by block from the bottom: a 32 x rem matrix-vector product by
//     128 threads, then the 32 x 32 triangle by one warp with its rows in registers (one shuffle
//     and one FMA per unknown).
// Measured and rejected (r02aa): per-warp staging pipelines (every warp copies its own slice of the
// pivot rows into its own two buffers, no block barrier in the accumulation loop) -- 336.6 against
// 309.4 ms per configs[2] epoch: 55 KB of shared memory per CTA instead of 36 (the L1 share of the SM
// shrinks from 92 to 28 KB at four CTAs) and twice the L2 reads for the duplicated diagonal-block
// columns cost more than the 13 % of stall samples at that barrier.
// Factor columns >= K (K < 256) are zero in P and G: their diagonal is set to 1, their solution
// is 0.  Failure rules of the reference: pivot not > 0 -> "Cholesky decomposition failed.",
// non-finite solution -> "Cholesky solve failed." (:316-323).
#include "common.cuh"

namespace ials {
namespace {

constexpr int kN = 256;            // order of the (padded) system = row stride of the factors
constexpr int kNB = 32;            // block row height
constexpr int kBlocks = kN / kNB;  // 8
constexpr int kLLThreads = 128;
constexpr int kStagePivots = 16;
constexpr int kStripLd = 232;  // staged rows: block rows p >= 1 are at most 224 + 8 floats wide
constexpr int kRowLd0 = 264;   // widest block row (p = 0): 256 columns + [z | 1 / U_kk | 0 x 6]

// scratch of one CTA: block row q = 32 rows of row_len(q) floats  [U(k, 32 q .. 255) | z_k | 1 / U_kk | 0 x 6]
__host__ __device__ constexpr int row_len(int q) { return kN - kNB * q + 8; }
__host__ __device__ constexpr int block_base(int q) { return 32 * (264 * q - 16 * q * (q - 1)); }
constexpr int kScratchFloats = block_base(kBlocks);  // 38 912

#define EL(i, j) (((j) & 1) ? acc[i][(j) >> 1].y : acc[i][(j) >> 1].x)
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) {
  float2 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;"
      : "=l"(*reinterpret_cast<unsigned long long *>(&d))
      : "l"(*reinterpret_cast<unsigned long long *>(&a)), "l"(*reinterpret_cast<unsigned long long *>(&b)),
        "l"(*reinterpret_cast<unsigned long long *>(&c)));
  return d;
}
// 16 bytes global -> shared at the same byte offset OFF from both base addresses (an immediate)
template <int OFF>
__device__ __forceinline__ void cp_async16_at(unsigned smem_addr, const void *gmem) {
  asm volatile("cp.async.cg.shared.global [%0 + %2], [%1 + %2], 16;" ::"r"(smem_addr), "l"(gmem), "n"(OFF)
               : "memory");
}
__device__ __forceinline__ void cp_async_commit_wait_all() {
  asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory");
}
__device__ __forceinline__ void prefetch_l2(const void *p) {
  asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
}

struct LLSmem {
  // two staged strips of a finished block row [2][16][kStripLd]  /  the current block row
  // [32][row_len(p)] between its accumulation and its factorisation  /  the triangle of the
  // back substitution
  float buf[kNB * kRowLd0];
  float rowbuf[2][kNB];  // the scaled pivot row of the diagonal block, double buffered
  float dinv[kNB];       // 1 / U_kk of the current block row
  float bpart[4][kNB];   // the warps' partial sums of the right-hand side
  float x[kN];           // solution
  float rs[kNB];         // right-hand side of the current triangle
  float sinv[kNB];
};
static_assert(2 * kStagePivots * kStripLd <= kNB * kRowLd0, "the strips alias the block row buffer");

// Workspace of one chunk of Gram jobs (solve.cu solve_cholesky_tensor, wgram.cu wgram256_kernel):
//   W [JC][256][256] | b [JC][kWGram256BParts][256];   G = W + W^T
struct LLArgs {
  const float *ws;
  int job0;        // first job of the chunk (row_jobs holds absolute job ids)
  int job_cap;     // JC
  float *scratch;  // [gridDim.x][kScratchFloats]
};

__global__ void __launch_bounds__(kLLThreads, 4) cholesky_ll_kernel(SolveArgs a, LLArgs g) {
  __shared__ __align__(16) LLSmem sm;
  __shared__ long long s_slot;
  __shared__ int s_fail;
  // (Rotating the warps' roles with the CTA's residency slot, so that every scheduler sees one
  // warp of each role instead of four warps of the same one, was measured and is 24 % SLOWER:
  // r02l, 21.0 against 17.0 ms per epoch at 5 % of configs[2].)
  const int tid = threadIdx.x, lane = tid % kWarp, warp = tid / kWarp;
  // tile (tr, tcr) of the block row; the four tiles of the right-hand side column are owned by
  // four threads of warp 0 whose own tiles lie below the diagonal (tid 1, 2, 3, 6), so the
  // column costs no instruction of its own
  int tr = tid & 3;
  const int tcr = tid >> 2;
  const bool rhs = tid == 1 || tid == 2 || tid == 3 || tid == 6;
  if (rhs) tr = tid == 6 ? 3 : tid - 1;
  const int K = a.K;
  float *const scratch = g.scratch + (size_t)blockIdx.x * kScratchFloats;
  const float *const wsb = g.ws + (size_t)g.job_cap * kN * kN;  // the b partials

  for (;;) {
    __syncthreads();
    if (tid == 0) {
      s_slot = (long long)atomicAdd(a.work_counter, 1ull);
      s_fail = 0;
    }
    __syncthreads();
    const int64_t slot = s_slot;
    if (slot >= a.n_sched) break;
    const int64_t u = a.order ? (int64_t)a.order[slot] : slot;
    const int64_t gu = a.row_base + u;
    const int64_t nnz = a.indptr[u + 1] - a.indptr[u];
    const float reg_u = a.reg * powf(a.alpha0 * (float)a.n_other + (float)nnz, a.nu);  // :309-310
    const int gj0 = a.row_jobs[slot] - g.job0, gj1 = a.row_jobs[slot + 1] - g.job0;
    bool failed = false;

    for (int p = 0; p < kBlocks; p++) {
      const int Wp = kN - kNB * p, Lp = Wp + 8, ntc = Wp / 8;
      const bool active = rhs || (tcr < ntc && (tcr >= 4 || tcr >= tr));
      const int colofs = rhs ? Wp : 8 * tcr;
      const int gi0 = kNB * p + 8 * tr, gjc = kNB * p + 8 * tcr;  // global row / column of the tile

      // b of the block row = the Gram producers' partial sums (:301-307): lane = row, a warp
      // takes two of the eight partials of every job (stored after the stages: the loads stay in
      // flight meanwhile)
      float bl = 0.f;
      {
        const float *bp = wsb + kNB * p + lane;
        for (int jb = gj0; jb < gj1; jb++)
#pragma unroll
          for (int q = 0; q < kWGram256BParts / 4; q++)
            bl += __ldcs(bp + ((size_t)jb * kWGram256BParts + (kWGram256BParts / 4) * warp + q) * kN);
      }
      // the tile's part of A (and of its mirror image): into L2 while the finished block rows
      // stream through
      if (active && !rhs && p > 0) {
        const float *W = g.ws + (size_t)gj0 * kN * kN;
#pragma unroll
        for (int i = 0; i < 8; i++) {
          prefetch_l2(a.P + (size_t)(gi0 + i) * kN + gjc);
          prefetch_l2(W + (size_t)(gi0 + i) * kN + gjc);
          prefetch_l2(W + (size_t)(gjc + i) * kN + gi0);
        }
      }

      float2 acc[8][4];
#pragma unroll
      for (int i = 0; i < 8; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) acc[i][j] = make_float2(0.f, 0.f);

      // ---- S = sum over the finished block rows, 16 pivots per stage ----
      const int n_stages = 2 * p, chunks_per_row = Lp / 4;
      // staging role of a thread: row tid / 8 of the stage, its 16-byte chunks tid % 8 + 8 i
      // (one address pair per stage and immediates after that: the first version divided the
      // chunk index by the row length, a loop over (warp, lane) strides ran 20 % more
      // instructions than even that -- r02k / r02n)
      const int n_chunks = (chunks_per_row - (tid & 7) + 7) >> 3;
      auto issue_stage = [&](int st) {
        const int q = st >> 1, k0 = kStagePivots * (st & 1);
        const float *src = scratch + block_base(q) + (size_t)(k0 + (tid >> 3)) * row_len(q) + kNB * (p - q) +
                           4 * (tid & 7);
        const unsigned dst = (unsigned)__cvta_generic_to_shared(
            sm.buf + (st & 1) * kStagePivots * kStripLd + (tid >> 3) * kStripLd + 4 * (tid & 7));
        if (0 < n_chunks) cp_async16_at<0>(dst, src);
        if (1 < n_chunks) cp_async16_at<128>(dst, src);
        if (2 < n_chunks) cp_async16_at<256>(dst, src);
        if (3 < n_chunks) cp_async16_at<384>(dst, src);
        if (4 < n_chunks) cp_async16_at<512>(dst, src);
        if (5 < n_chunks) cp_async16_at<640>(dst, src);
        if (6 < n_chunks) cp_async16_at<768>(dst, src);
        if (7 < n_chunks) cp_async16_at<896>(dst, src);
      };
      if (n_stages > 0) issue_stage(0);
      for (int st = 0; st < n_stages; st++) {
        cp_async_commit_wait_all();
        __syncthreads();  // stage st has landed; everybody is done with the other buffer
        if (st + 1 < n_stages) issue_stage(st + 1);
        if (active) {
          const float *sb = sm.buf + (st & 1) * kStagePivots * kStripLd;
#pragma unroll 4
          for (int k = 0; k < kStagePivots; k++) {
            const float4 r0 = *reinterpret_cast<const float4 *>(sb + k * kStripLd + 8 * tr);
            const float4 r1 = *reinterpret_cast<const float4 *>(sb + k * kStripLd + 8 * tr + 4);
            const float4 c0 = *reinterpret_cast<const float4 *>(sb + k * kStripLd + colofs);
            const float4 c1 = *reinterpret_cast<const float4 *>(sb + k * kStripLd + colofs + 4);
            const float ra[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
            const float2 cb[4] = {make_float2(c0.x, c0.y), make_float2(c0.z, c0.w), make_float2(c1.x, c1.y),
                                  make_float2(c1.z, c1.w)};
#pragma unroll
            for (int i = 0; i < 8; i++)
#pragma unroll
              for (int j = 0; j < 4; j++) acc[i][j] = fma2(make_float2(ra[i], ra[i]), cb[j], acc[i][j]);
          }
        }
      }
      sm.bpart[warp][lane] = bl;
      __syncthreads();  // the strips are consumed (the block row goes into the same buffer); b is complete

      // ---- acc = A - S ----
      if (rhs) {
#pragma unroll
        for (int i = 0; i < 8; i++) {
          const int r = 8 * tr + i;
          EL(i, 0) = ((sm.bpart[0][r] + sm.bpart[1][r]) + (sm.bpart[2][r] + sm.bpart[3][r])) - EL(i, 0);
        }
      } else if (active) {
#pragma unroll
        for (int i = 0; i < 8; i++) {
          const float4 p0 = *reinterpret_cast<const float4 *>(a.P + (size_t)(gi0 + i) * kN + gjc);
          const float4 p1 = *reinterpret_cast<const float4 *>(a.P + (size_t)(gi0 + i) * kN + gjc + 4);
          acc[i][0] = make_float2(p0.x - acc[i][0].x, p0.y - acc[i][0].y);
          acc[i][1] = make_float2(p0.z - acc[i][1].x, p0.w - acc[i][1].y);
          acc[i][2] = make_float2(p1.x - acc[i][2].x, p1.y - acc[i][2].y);
          acc[i][3] = make_float2(p1.z - acc[i][3].x, p1.w - acc[i][3].y);
        }
        for (int jb = gj0; jb < gj1; jb++) {
          const float *W = g.ws + (size_t)jb * kN * kN;
#pragma unroll
          for (int i = 0; i < 8; i++) {
            const float4 w0 = __ldcs(reinterpret_cast<const float4 *>(W + (size_t)(gi0 + i) * kN + gjc));
            const float4 w1 = __ldcs(reinterpret_cast<const float4 *>(W + (size_t)(gi0 + i) * kN + gjc + 4));
            acc[i][0].x += w0.x; acc[i][0].y += w0.y; acc[i][1].x += w0.z; acc[i][1].y += w0.w;
            acc[i][2].x += w1.x; acc[i][2].y += w1.y; acc[i][3].x += w1.z; acc[i][3].y += w1.w;
          }
#pragma unroll
          for (int j = 0; j < 8; j++) {  // + W^T: row gjc + j of W holds column j of the tile
            const float4 w0 = __ldcs(reinterpret_cast<const float4 *>(W + (size_t)(gjc + j) * kN + gi0));
            const float4 w1 = __ldcs(reinterpret_cast<const float4 *>(W + (size_t)(gjc + j) * kN + gi0 + 4));
            EL(0, j) += w0.x; EL(1, j) += w0.y; EL(2, j) += w0.z; EL(3, j) += w0.w;
            EL(4, j) += w1.x; EL(5, j) += w1.y; EL(6, j) += w1.z; EL(7, j) += w1.w;
          }
        }
        if (gi0 == gjc) {  // :312-314; the padding columns get a unit diagonal
#pragma unroll
          for (int i = 0; i < 8; i++) {
            if (gi0 + i < K) EL(i, i) += reg_u;
            else EL(i, i) = 1.f;
          }
        }
      }

      // ---- the block row itself.  The tiles go to shared memory; warp 0 factors the 32 x 32
      // diagonal block (lane = column); then every thread owns two whole COLUMNS of the panel
      // and solves them against the triangle: no barrier and no divergence inside either phase
      // (r02j ncu: the tile-row formulation spent 48 % of its stall samples at its 8 block
      // barriers and executed 78 k of the row's 236 k warp instructions in half-empty warps).
      float *const brow = sm.buf;  // [32][Lp]
      if (active) {
#pragma unroll
        for (int i = 0; i < 8; i++) {
          float *dst = brow + (8 * tr + i) * Lp + colofs;
          *reinterpret_cast<float4 *>(dst) = make_float4(acc[i][0].x, acc[i][0].y, acc[i][1].x, acc[i][1].y);
          *reinterpret_cast<float4 *>(dst + 4) = make_float4(acc[i][2].x, acc[i][2].y, acc[i][3].x, acc[i][3].y);
        }
      }
      __syncthreads();
      float *const gblock = scratch + block_base(p);
      if (warp == 0) {
        float col[kNB];  // col[i] = A(i, lane), meaningful for i <= lane
#pragma unroll
        for (int i = 0; i < kNB; i++) col[i] = brow[i * Lp + lane];
        bool bad = false;
        float akk = __shfl_sync(0xffffffffu, col[0], 0);
#pragma unroll
        for (int k = 0; k < kNB; k++) {
          bad = bad || !(akk > 0.f);
          const float inv = __frsqrt_rn(akk);
          const float ukj = col[k] * inv;  // U(k, lane) for lane >= k
          col[k] = ukj;
          // the next pivot is lane k + 1's own business (a - sum of ITS squares): it is on its way
          // to the other lanes while the pivot row makes its round trip through shared memory --
          // the chain pivot -> rsqrt -> scale -> next pivot no longer waits for that round trip
          if (k + 1 < kNB) akk = __shfl_sync(0xffffffffu, fmaf(-ukj, ukj, col[k + 1]), k + 1);
          float *rb = sm.rowbuf[k & 1];
          rb[lane] = ukj;
          if (lane == k) sm.dinv[k] = inv;
          __syncwarp();
          // trailing update of the upper triangle: A(i, lane) -= U(k, i) U(k, lane), k < i <= lane
          // (entries below the diagonal and the lanes left of k compute values nobody reads)
#pragma unroll
          for (int i4 = (k + 1) / 4; i4 < kNB / 4; i4++) {
            const float4 r = *reinterpret_cast<const float4 *>(rb + 4 * i4);
            if (4 * i4 + 0 > k) col[4 * i4 + 0] = fmaf(-r.x, ukj, col[4 * i4 + 0]);
            if (4 * i4 + 1 > k) col[4 * i4 + 1] = fmaf(-r.y, ukj, col[4 * i4 + 1]);
            if (4 * i4 + 2 > k) col[4 * i4 + 2] = fmaf(-r.z, ukj, col[4 * i4 + 2]);
            if (4 * i4 + 3 > k) col[4 * i4 + 3] = fmaf(-r.w, ukj, col[4 * i4 + 3]);
          }
        }
        if (bad && lane == 0) s_fail = 1;
        // the triangle, zero below the diagonal: to shared memory for the panel, to the scratch
#pragma unroll
        for (int k = 0; k < kNB; k++) {
          const float v = k <= lane ? col[k] : 0.f;
          brow[k * Lp + lane] = v;
          gblock[(size_t)k * Lp + lane] = v;
        }
        gblock[(size_t)lane * Lp + Wp + 1] = sm.dinv[lane];  // own write above (lane == k)
      }
      __syncthreads();
      if (s_fail) {  // uniform: written before the barrier every thread just passed
        failed = true;
        break;
      }
      {
        // panel column c <-> block row column 32 + c; the last one (c = Wp - 32) is the
        // right-hand side: its solution is z.  Two columns per thread, packed.
        const int ncol = Wp - kNB + 1;
        const int ca = tid, cb2 = tid + kLLThreads;
        if (ca < ncol) {
          const bool two = cb2 < ncol;
          float2 z[kNB];
#pragma unroll
          for (int i = 0; i < kNB; i++)
            z[i] = make_float2(brow[i * Lp + kNB + ca], two ? brow[i * Lp + kNB + cb2] : 0.f);
#pragma unroll
          for (int k = 0; k < kNB; k++) {
            const float inv = sm.dinv[k];
            z[k] = make_float2(z[k].x * inv, z[k].y * inv);
#pragma unroll
            for (int i4 = (k + 1) / 4; i4 < kNB / 4; i4++) {
              const float4 r = *reinterpret_cast<const float4 *>(brow + k * Lp + 4 * i4);  // U(k, 4 i4 ..)
              if (4 * i4 + 0 > k) z[4 * i4 + 0] = fma2(make_float2(-r.x, -r.x), z[k], z[4 * i4 + 0]);
              if (4 * i4 + 1 > k) z[4 * i4 + 1] = fma2(make_float2(-r.y, -r.y), z[k], z[4 * i4 + 1]);
              if (4 * i4 + 2 > k) z[4 * i4 + 2] = fma2(make_float2(-r.z, -r.z), z[k], z[4 * i4 + 2]);
              if (4 * i4 + 3 > k) z[4 * i4 + 3] = fma2(make_float2(-r.w, -r.w), z[k], z[4 * i4 + 3]);
            }
          }
#pragma unroll
          for (int k = 0; k < kNB; k++) {
            gblock[(size_t)k * Lp + kNB + ca] = z[k].x;
            if (two) gblock[(size_t)k * Lp + kNB + cb2] = z[k].y;
          }
        }
      }
      __syncthreads();  // the block row is in the scratch; its shared-memory copy may be overwritten
    }
    if (failed) {
      if (tid == 0) atomicExch(&a.err_flags[kErrCholDecomp], 1);
      continue;
    }

    // ---- backward substitution  U x = z, block by block from the bottom ----
    for (int p = kBlocks - 1; p >= 0; p--) {
      const int Wp = kN - kNB * p, Lp = Wp + 8;
      const float *Ub = scratch + block_base(p);
      {  // 4 threads per row: z - U(row, columns right of the diagonal block) . x
        const int row = tid >> 2, part = tid & 3;
        const float *Ur = Ub + (size_t)row * Lp;
        float dot = 0.f;
        for (int c4 = kNB / 4 + part; c4 < Wp / 4; c4 += 4) {
          const float4 uv = __ldcg(reinterpret_cast<const float4 *>(Ur + 4 * c4));
          const float4 xv = *reinterpret_cast<const float4 *>(&sm.x[kNB * p + 4 * c4]);
          dot = fmaf(uv.x, xv.x, dot);
          dot = fmaf(uv.y, xv.y, dot);
          dot = fmaf(uv.z, xv.z, dot);
          dot = fmaf(uv.w, xv.w, dot);
        }
        dot += __shfl_xor_sync(0xffffffffu, dot, 1);
        dot += __shfl_xor_sync(0xffffffffu, dot, 2);
        if (part == 0) {
          sm.rs[row] = __ldcg(Ur + Wp) - dot;
          sm.sinv[row] = __ldcg(Ur + Wp + 1);
        }
        // the triangle, padded to 33 floats per row
        const float4 t0 = __ldcg(reinterpret_cast<const float4 *>(Ur + 8 * part));
        const float4 t1 = __ldcg(reinterpret_cast<const float4 *>(Ur + 8 * part + 4));
        float *td = sm.buf + row * 33 + 8 * part;
        td[0] = t0.x; td[1] = t0.y; td[2] = t0.z; td[3] = t0.w;
        td[4] = t1.x; td[5] = t1.y; td[6] = t1.z; td[7] = t1.w;
      }
      __syncthreads();
      if (warp == 0) {  // lane = row j of the triangle, its 32 entries in registers
        const float *tri = sm.buf + lane * 33;
        float ur[kNB];
#pragma unroll
        for (int i = 0; i < kNB; i++) ur[i] = tri[i];
        float r = sm.rs[lane];
        const float inv = sm.sinv[lane];
        float xmine = 0.f;
#pragma unroll
        for (int i = kNB - 1; i >= 0; i--) {
          const float xi = __shfl_sync(0xffffffffu, r * inv, i);
          if (lane == i) xmine = xi;
          if (lane < i) r = fmaf(-ur[i], xi, r);
        }
        sm.x[kNB * p + lane] = xmine;
      }
      __syncthreads();
    }
    bool finite = true;
    for (int k = tid; k < K; k += kLLThreads) finite = finite && isfinite(sm.x[k]);
    if (!finite) s_fail = 1;
    __syncthreads();
    if (s_fail) {  // :320-323
      if (tid == 0) atomicExch(&a.err_flags[kErrCholSolve], 1);
      continue;
    }
    for (int k = tid; k < kN; k += kLLThreads) {
      const float v = k < K ? sm.x[k] : 0.f;
      a.target[gu * kN + k] = v;
      for (int pi = 0; pi < a.n_peers; pi++) a.peers[pi][gu * kN + k] = v;
    }
  }
}

}  // namespace

// resident CTAs of cholesky_ll_kernel on the current device and its scratch size
static int ll_grid() {
  int dev = 0, sms = kNumSMsB200, per_sm = 0;
  CUDA_CHECK(cudaGetDevice(&dev));
  CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, cholesky_ll_kernel, kLLThreads, 0));
  return sms * std::max(per_sm, 1);
}
size_t cholesky_ll_scratch_bytes() { return (size_t)ll_grid() * kScratchFloats * sizeof(float); }

// Cholesky rows whose Gram blocks are in `workspace`: a.order / a.n_sched = the chunk's rows,
// first_job[0 .. n_sched] their absolute job ranges, scratch >= cholesky_ll_scratch_bytes().
void launch_solve_cholesky_from_gram(const SolveArgs &a, const int32_t *first_job, int job0, int job_cap,
                                     const float *workspace, float *scratch, cudaStream_t s) {
  if (a.n_sched <= 0) return;
  if (a.ld != kN || a.K > kN) throw NotImplemented("Cholesky from Gram blocks: the row stride must be 256");
  SolveArgs args = a;
  args.row_jobs = first_job;
  CUDA_CHECK(cudaMemsetAsync(a.work_counter, 0, sizeof(unsigned long long), s));
  const unsigned grid = (unsigned)std::min<int64_t>(a.n_sched, ll_grid());
  cholesky_ll_kernel<<<grid, kLLThreads, 0, s>>>(args, LLArgs{workspace, job0, job_cap, scratch});
  count_launch();
  CUDA_CHECK(cudaGetLastError());
}

}  // namespace ials
