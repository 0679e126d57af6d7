// Weighted, gathered Gram on the 5th-generation tensor cores (tcgen05 + TMEM):
//
//     G_job = sum_{t in job} w_t * y_{i_t} y_{i_t}^T          (128 x 128 block of a K x K matrix)
//
// One kernel, three callers:
//   * K1  Solver::prepare_p                 P = alpha0 * Y^T Y   (all rows, w = 1)
//         /root/reference/cpp_source/als/IALSTrainer.hpp:78-115
//   * K2  heavy rows of Solver::step_cg     A_u = P + reg_u I + sum c y y^T formed explicitly
//         (:216-247 evaluate the same operator neighbour by neighbour)
//   * K3  Solver::step_cholesky's rank update for 256-column factors (BatchedRankUpdater,
//         :37-58, 301-308): wgram256_kernel below, the same scheme on 256 x 256.
//
// float32 parity on TF32 tensor cores: u = sqrt(w) * y is split into hi = tf32(u) and
// lo = u - hi (exact), and  u u^T = hi hi^T + hi lo^T + lo hi^T + O(2^-22).  The
// kernel accumulates  HH = sum hi hi^T  and  HL = sum hi lo^T  in two TMEM accumulators (fp32,
// one N = 256 MMA per 8 neighbours with [hi | lo] as the B operand) and emits  W = HH / 2 + HL;
// consumers use  G = W + W^T,  which is exactly symmetric.
//
// Structure (one persistent CTA per SM, 672 threads):
//   warps 0-15  producers (four groups of four warps, round-robin over the stages): a warp owns 8
//               CONSECUTIVE neighbours of the stage and a lane the features {l, l+32, l+64, l+96}:
//               four coalesced 128-byte LDG.32 per neighbour, then the 8 neighbours of one feature
//               sit in one lane's registers and leave as two conflict-free STS.128 per tile into
//               the canonical K-major SWIZZLE_128B layout (tc.cuh desc_kmajor_sw128: a tile row is
//               one feature, 128 bytes = the stage's 32 neighbours); also b = sum (bias + w) y.
//   warp  20    MMA issuer: one elected lane issues tcgen05.mma.kind::tf32 (M = 128, N = 256,
//               K = 8) and tcgen05.commit to the stage / accumulator barriers.
//   warps 16-19 epilogue: tcgen05.ld the two accumulators (double-buffered: 2 x 256 TMEM columns),
//               combine, and write W to global memory.
// Stages: 4 x (128 features x 32 neighbours x (hi + lo)) = 128 KB of shared memory.
// Measured (r02a, tools/time_wgram.py before its removal): 20.7 ns per neighbour and SM against
// 21.7 ns for the MN-major operand layout of round 1 (deleted); the producers (gather +
// conversion, 19.7 ns without the MMA) and the barrier handshakes (9.4 ns with nothing else)
// bound it, not the tensor pipe (15.1 ns with the producers idle).  Two producer groups of four
// warps with the gather of a group's next stage in flight during the conversion (the scoring
// kernel's scheme) were measured in r02p: 33 ns per neighbour -- the conversion needs the sixteen
// warps' worth of independent instruction streams more than the gather needs slack.
#include "common.cuh"
#include "tc.cuh"

namespace ials {
namespace {

using namespace tc;

constexpr int KP = 128;
constexpr int KT = 32;  // neighbours per stage = one 128-byte K-major row of tf32
constexpr int STAGES = 4;
constexpr int kProducerWarps = 4;
constexpr int kGroups = 4;
constexpr int kAllProducerWarps = kGroups * kProducerWarps;
static_assert(kAllProducerWarps == kWGramBParts, "bpart layout");
constexpr int kEpilogueWarps = 4;
constexpr int kThreads = (kAllProducerWarps + kEpilogueWarps + 1) * kWarp;
constexpr int kTileBytes = KP * 128;          // 16 KB: hi or lo, 128 feature rows x 32 neighbours
constexpr int kStageBytes = 2 * kTileBytes;   // 32 KB
constexpr int kTmemCols = 512;
constexpr uint32_t kIdesc = idesc_tf32(KP, 2 * KP, false, false);  // both operands K-major

// 16-byte store to a shared-window address (STS.128; a float4 store through the generic pointer
// derived from the aligned dynamic-shared base compiles to generic ST.E pieces)
__device__ __forceinline__ void sts4(uint32_t addr, float x, float y, float z, float w) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(x), "f"(y), "f"(z), "f"(w)
               : "memory");
}

struct StageCursor {  // as in wgram.cu
  int j, base, je;
  unsigned it;
  __device__ __forceinline__ bool valid(const WGramArgs &a) const { return j < (int)a.n_jobs; }
  __device__ __forceinline__ void seek(const WGramArgs &a, int grid) {
    base = je = 0;
    while (j < (int)a.n_jobs) {
      base = (int)a.job_begin[j];
      je = (int)a.job_end[j];
      if (je > base) return;
      j += grid;
    }
  }
  __device__ __forceinline__ void advance(const WGramArgs &a, int grid) {
    base += KT;
    it++;
    if (base >= je) {
      j += grid;
      seek(a, grid);
    }
  }
};

__global__ void __launch_bounds__(kThreads, 1) wgram_kernel(WGramArgs a) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char *tiles = reinterpret_cast<unsigned char *>(
      ((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t *bars = reinterpret_cast<uint64_t *>(tiles + STAGES * kStageBytes);
  uint64_t *full = bars;
  uint64_t *empty = bars + STAGES;
  uint64_t *accfull = bars + 2 * STAGES;
  uint64_t *accempty = accfull + 2;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(accempty + 2);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (tid == 0) {
    for (int s = 0; s < STAGES; s++) {
      mbar_init(&full[s], kProducerWarps);
      mbar_init(&empty[s], 1);
    }
    for (int b = 0; b < 2; b++) {
      mbar_init(&accfull[b], 1);
      mbar_init(&accempty[b], kEpilogueWarps);
    }
    mbar_init_fence();
  }
  if (warp == kAllProducerWarps + kEpilogueWarps) tmem_alloc(tmem_slot, kTmemCols);
  fence_before();
  __syncthreads();
  fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < kAllProducerWarps) {
    // ================================ PRODUCERS ================================
    const int group = warp / kProducerWarps, pw = warp % kProducerWarps;
    const int grid = (int)gridDim.x;
    int flushed = (int)blockIdx.x - grid;
    float bacc[4] = {0.f, 0.f, 0.f, 0.f};  // features lane + 32 j
    auto flush_until = [&](int j_stop) {
      for (int jj = flushed + grid; jj < j_stop && jj < (int)a.n_jobs; jj += grid) {
        if (a.bpart) {
          float *dst = a.bpart + ((size_t)jj * kAllProducerWarps + warp) * KP + lane;
#pragma unroll
          for (int j = 0; j < 4; j++) dst[32 * j] = bacc[j];
        }
#pragma unroll
        for (int j = 0; j < 4; j++) bacc[j] = 0.f;
        flushed = jj;
      }
    };
    auto next_own = [&](StageCursor c) {
      for (int g = 0; g < kGroups && c.valid(a); g++) c.advance(a, grid);
      return c;
    };
    auto load_ids = [&](const StageCursor &c, int &row, float &w) {  // one neighbour per lane
      row = 0;
      w = 0.f;
      if (c.valid(a) && c.base + lane < c.je) {
        row = a.indices ? a.indices[c.base + lane] : c.base + lane;
        w = a.weights ? a.weights[c.base + lane] : 1.f;
      }
    };
    StageCursor cur;
    cur.j = (int)blockIdx.x;
    cur.it = 0;
    cur.seek(a, grid);
    for (int g = 0; g < group && cur.valid(a); g++) cur.advance(a, grid);
    StageCursor n1 = next_own(cur), n2 = next_own(n1);
    int row0, row1, row2;
    float w0, w1, w2;
    load_ids(cur, row0, w0);
    load_ids(n1, row1, w1);
    load_ids(n2, row2, w2);
    constexpr int NPW = KT / kProducerWarps;  // 8 consecutive neighbours per warp and stage
    static_assert(NPW == 8, "two 16-byte chunks of four neighbours per feature row");
    while (cur.valid(a)) {
      flush_until(cur.j);
      const int s = (int)(cur.it % STAGES);
      const uint32_t ph = (uint32_t)((cur.it / STAGES) & 1);
      const int m = min(KT, cur.je - cur.base);
      float v[NPW][4];
#pragma unroll
      for (int q = 0; q < NPW; q++) {
        const int t = NPW * pw + q;
        const int row = __shfl_sync(0xffffffffu, row0, t);
        const float *src = a.Y + (size_t)row * a.ld + lane;
#pragma unroll
        for (int j = 0; j < 4; j++) v[q][j] = t < m ? __ldg(src + 32 * j) : 0.f;
      }
      const StageCursor n3 = next_own(n2);
      int row3;
      float w3;
      load_ids(n3, row3, w3);

      mbar_wait(&empty[s], ph ^ 1);
      const uint32_t hi = smem_u32(tiles + s * kStageBytes), lo = hi + kTileBytes;
      float sc[NPW];
#pragma unroll
      for (int q = 0; q < NPW; q++) {
        const int t = NPW * pw + q;
        const float w = __shfl_sync(0xffffffffu, w0, t);
        sc[q] = sqrtf(fmaxf(w, 0.f));
        const float cb = t < m ? a.bias + w : 0.f;
#pragma unroll
        for (int j = 0; j < 4; j++) bacc[j] = fmaf(cb, v[q][j], bacc[j]);
      }
#pragma unroll
      for (int j = 0; j < 4; j++) {
        const int f = lane + 32 * j;  // tile row = feature
#pragma unroll
        for (int half = 0; half < 2; half++) {
          float h[4], l[4];
#pragma unroll
          for (int e = 0; e < 4; e++) {
            const int q = 4 * half + e;
            const float u = sc[q] * v[q][j];
            h[e] = __uint_as_float(__float_as_uint(u) & 0xffffe000u);
            l[e] = u - h[e];
          }
          const uint32_t off = sw128_offset(f, 2 * pw + half);  // 16-byte chunk = 4 neighbours
          sts4(hi + off, h[0], h[1], h[2], h[3]);
          sts4(lo + off, l[0], l[1], l[2], l[3]);
        }
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&full[s]);
      cur = n1; n1 = n2; n2 = n3;
      row0 = row1; row1 = row2; row2 = row3;
      w0 = w1; w1 = w2; w2 = w3;
    }
    flush_until((int)a.n_jobs);
  } else if (warp == kAllProducerWarps + kEpilogueWarps) {
    // ================================ MMA ISSUER ================================
    unsigned long long it = 0, jc = 0;
    for (long long j = blockIdx.x; j < a.n_jobs; j += gridDim.x) {
      const long long jb = a.job_begin[j], je = a.job_end[j];
      if (je <= jb) continue;
      const int buf = (int)(jc & 1);
      mbar_wait(&accempty[buf], (uint32_t)(((jc >> 1) & 1) ^ 1));
      fence_after();
      const uint32_t d = tmem_base + (uint32_t)(buf * 256);
      uint32_t acc = 0;
      for (long long base = jb; base < je; base += KT, it++) {
        const int s = (int)(it % STAGES);
        mbar_wait(&full[s], (uint32_t)((it / STAGES) & 1));
        fence_after();
        if (lane == 0) {
          const uint32_t hi = smem_u32(tiles + s * kStageBytes);
#pragma unroll
          for (int k = 0; k < KT / 8; k++) {
            // A = hi rows 0..127, B = rows 0..255 of the stage ([hi | lo]); 8 neighbours = 32 bytes
            const uint64_t dh = desc_kmajor_sw128(hi + k * 32);
            mma_tf32(d, dh, dh, acc, kIdesc);
            acc = 1;
          }
          commit(&empty[s]);
          if (base + KT >= je) commit(&accfull[buf]);
        }
        __syncwarp();
      }
      jc++;
    }
  } else {
    // ================================ EPILOGUE ================================
    const int ew = warp - kAllProducerWarps;
    const int row = ew * 32 + lane;
    unsigned long long jc = 0;
    for (long long j = blockIdx.x; j < a.n_jobs; j += gridDim.x) {
      float *out = a.W + (size_t)j * KP * KP + (size_t)row * KP;
      if (a.job_end[j] <= a.job_begin[j]) {
#pragma unroll 4
        for (int c = 0; c < KP; c += 4) *reinterpret_cast<float4 *>(out + c) = make_float4(0.f, 0.f, 0.f, 0.f);
        continue;
      }
      const int buf = (int)(jc & 1);
      mbar_wait(&accfull[buf], (uint32_t)((jc >> 1) & 1));
      fence_after();
      const uint32_t t_hh = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(buf * 256);
#pragma unroll 1
      for (int c = 0; c < KP; c += 16) {
        uint32_t hh[16], hl[16];
        tmem_ld16(t_hh + c, hh);
        tmem_ld16(t_hh + 128 + c, hl);
        tmem_ld_wait();
#pragma unroll
        for (int q = 0; q < 16; q += 4) {
          float4 o;
          o.x = fmaf(0.5f, __uint_as_float(hh[q + 0]), __uint_as_float(hl[q + 0]));
          o.y = fmaf(0.5f, __uint_as_float(hh[q + 1]), __uint_as_float(hl[q + 1]));
          o.z = fmaf(0.5f, __uint_as_float(hh[q + 2]), __uint_as_float(hl[q + 2]));
          o.w = fmaf(0.5f, __uint_as_float(hh[q + 3]), __uint_as_float(hl[q + 3]));
          *reinterpret_cast<float4 *>(out + c + q) = o;
        }
      }
      fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&accempty[buf]);
      jc++;
    }
  }

  fence_before();
  __syncthreads();
  if (warp == kAllProducerWarps + kEpilogueWarps) tmem_dealloc(tmem_base, kTmemCols);
}


// ---------------------------------------------------------------------------------------------
// Whole Gram of 256-column factor rows in ONE pass over the neighbours (K = 256 Cholesky,
// BASELINE configs[2]; solve.cu solve_cholesky_tensor).  A 256-float row is two halves y0 | y1;
// with u = sqrt(c) y = hi + lo as above,
//     W = 1/2 hi (hi + 2 lo)^T      (256 x 256),        G = sum c y y^T = W + W^T + O(2^-22)
// (W + W^T = hi hi^T + hi lo^T + lo hi^T; 2 lo is as exact in TF32 as lo).  A stage holds four
// K-major tiles [hi0 | hi1 | 2 lo0 | 2 lo1] (64 KB, 3 stages), so both B operands are 256
// contiguous tile rows, and per 8 neighbours four N = 256 instructions fill the two accumulators
//     D_top (rows   0..127) += hi0 x [hi0 | hi1]^T,   += hi0 x [2 lo0 | 2 lo1]^T
//     D_bot (rows 128..255) += hi1 x [hi0 | hi1]^T,   += hi1 x [2 lo0 | 2 lo1]^T
// = all 512 TMEM columns: the epilogue of a job and the MMAs of the next do not overlap, and the
// large and the small products share an accumulator (two truncating fp32 accumulations per 8
// neighbours instead of one: tests/test_wgram.py states the tolerance that follows).
// Round 2 first ran three launches per chunk (this file's wgram_kernel on Y and on Y + 128 plus
// a cross-block kernel): three gathers of every neighbour row (2 KB for 1 KB) and three
// pipelines' worth of stage handshakes -- 114 ns per neighbour and SM on the full Netflix shape
// (r02k) against 34 ns of tensor time for the instructions above; this kernel: 56 ns on the long
// item rows (r02n).
//
// Producer groups = 2 <= stages = 3: a group waits for "its" slot with a phase-parity test,
// which is only sound while the slot's barrier is at most one phase behind what the group waits
// for; with G groups round-robin over S stages that holds iff G <= S (four groups over three
// stages deadlocked the cross-block kernel from a few thousand jobs on, r02b / r02g).
// 13 warps: 8 producers (a warp = 8 neighbours x 256 features of the stage in registers,
// 128 registers per thread), 4 epilogue, 1 MMA issuer.
// ---------------------------------------------------------------------------------------------
constexpr int YSTAGES = 3;
constexpr int kYGroups = 2;
constexpr int kYProducerWarps = kYGroups * kProducerWarps;
static_assert(kYProducerWarps == kWGram256BParts, "bpart layout");
static_assert(kYGroups <= YSTAGES, "phase-parity waits need groups <= stages");
constexpr int kYThreads = (kYProducerWarps + kEpilogueWarps + 1) * kWarp;  // 416
constexpr int kYStageBytes = 4 * kTileBytes;                               // 64 KB
constexpr int KY = 2 * KP;                                                 // 256 features

__global__ void __launch_bounds__(kYThreads, 1) wgram256_kernel(WGramArgs a) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char *tiles = reinterpret_cast<unsigned char *>(
      ((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t *bars = reinterpret_cast<uint64_t *>(tiles + YSTAGES * kYStageBytes);
  uint64_t *full = bars;               // [YSTAGES]
  uint64_t *empty = bars + YSTAGES;    // [YSTAGES]
  uint64_t *accfull = bars + 2 * YSTAGES;
  uint64_t *accempty = accfull + 1;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(accempty + 1);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  constexpr int kMmaWarp = kYProducerWarps + kEpilogueWarps;

  if (tid == 0) {
    for (int s = 0; s < YSTAGES; s++) {
      mbar_init(&full[s], kProducerWarps);
      mbar_init(&empty[s], 1);
    }
    mbar_init(accfull, 1);
    mbar_init(accempty, kEpilogueWarps);
    mbar_init_fence();
  }
  if (warp == kMmaWarp) tmem_alloc(tmem_slot, kTmemCols);
  fence_before();
  __syncthreads();
  fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < kYProducerWarps) {
    // ================================ PRODUCERS ================================
    const int group = warp / kProducerWarps, pw = warp % kProducerWarps;
    const int grid = (int)gridDim.x;
    int flushed = (int)blockIdx.x - grid;
    float bacc[8];  // features lane + 32 j
#pragma unroll
    for (int j = 0; j < 8; j++) bacc[j] = 0.f;
    auto flush_until = [&](int j_stop) {
      for (int jj = flushed + grid; jj < j_stop && jj < (int)a.n_jobs; jj += grid) {
        if (a.bpart) {
          float *dst = a.bpart + ((size_t)jj * kYProducerWarps + warp) * KY + lane;
#pragma unroll
          for (int j = 0; j < 8; j++) dst[32 * j] = bacc[j];
        }
#pragma unroll
        for (int j = 0; j < 8; j++) bacc[j] = 0.f;
        flushed = jj;
      }
    };
    auto next_own = [&](StageCursor c) {
      for (int g = 0; g < kYGroups && c.valid(a); g++) c.advance(a, grid);
      return c;
    };
    auto load_ids = [&](const StageCursor &c, int &row, float &w) {  // one neighbour per lane
      row = 0;
      w = 0.f;
      if (c.valid(a) && c.base + lane < c.je) {
        row = a.indices ? a.indices[c.base + lane] : c.base + lane;
        w = a.weights ? a.weights[c.base + lane] : 1.f;
      }
    };
    StageCursor cur;
    cur.j = (int)blockIdx.x;
    cur.it = 0;
    cur.seek(a, grid);
    for (int g = 0; g < group && cur.valid(a); g++) cur.advance(a, grid);
    StageCursor n1 = next_own(cur);
    int row0, row1;
    float w0, w1;
    load_ids(cur, row0, w0);
    load_ids(n1, row1, w1);
    constexpr int NPW = KT / kProducerWarps;  // 8 consecutive neighbours per warp and stage
    while (cur.valid(a)) {
      flush_until(cur.j);
      const int s = (int)(cur.it % YSTAGES);
      const uint32_t ph = (uint32_t)((cur.it / YSTAGES) & 1);
      const int m = min(KT, cur.je - cur.base);
      float v[NPW][8];
#pragma unroll
      for (int q = 0; q < NPW; q++) {
        const int t = NPW * pw + q;
        const int row = __shfl_sync(0xffffffffu, row0, t);
        const float *src = a.Y + (size_t)row * a.ld + lane;
#pragma unroll
        for (int j = 0; j < 8; j++) v[q][j] = t < m ? __ldg(src + 32 * j) : 0.f;
      }
      const StageCursor n2 = next_own(n1);
      int row2;
      float w2;
      load_ids(n2, row2, w2);
      float sc[NPW];
#pragma unroll
      for (int q = 0; q < NPW; q++) {
        const int t = NPW * pw + q;
        const float w = __shfl_sync(0xffffffffu, w0, t);
        sc[q] = sqrtf(fmaxf(w, 0.f));
        const float cb = t < m ? a.bias + w : 0.f;
#pragma unroll
        for (int j = 0; j < 8; j++) bacc[j] = fmaf(cb, v[q][j], bacc[j]);
      }
      mbar_wait(&empty[s], ph ^ 1);
      const uint32_t st = smem_u32(tiles + s * kYStageBytes);
#pragma unroll
      for (int j = 0; j < 8; j++) {
        const int f = lane + 32 * (j & 3);  // tile row = feature within its half
        const uint32_t hi = st + (uint32_t)(j >> 2) * kTileBytes, lo = hi + 2 * kTileBytes;
#pragma unroll
        for (int half = 0; half < 2; half++) {
          float h[4], l[4];
#pragma unroll
          for (int e = 0; e < 4; e++) {
            const int q = 4 * half + e;
            const float u = sc[q] * v[q][j];
            h[e] = __uint_as_float(__float_as_uint(u) & 0xffffe000u);
            l[e] = 2.f * (u - h[e]);
          }
          const uint32_t off = sw128_offset(f, 2 * pw + half);  // 16-byte chunk = 4 neighbours
          sts4(hi + off, h[0], h[1], h[2], h[3]);
          sts4(lo + off, l[0], l[1], l[2], l[3]);
        }
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&full[s]);
      cur = n1; n1 = n2;
      row0 = row1; row1 = row2;
      w0 = w1; w1 = w2;
    }
    flush_until((int)a.n_jobs);
  } else if (warp == kMmaWarp) {
    // ================================ MMA ISSUER ================================
    unsigned long long it = 0, jc = 0;
    for (long long j = blockIdx.x; j < a.n_jobs; j += gridDim.x) {
      const long long jb = a.job_begin[j], je = a.job_end[j];
      if (je <= jb) continue;
      mbar_wait(accempty, (uint32_t)((jc & 1) ^ 1));
      fence_after();
      uint32_t acc = 0;
      for (long long base = jb; base < je; base += KT, it++) {
        const int s = (int)(it % YSTAGES);
        mbar_wait(&full[s], (uint32_t)((it / YSTAGES) & 1));
        fence_after();
        if (lane == 0) {
          const uint32_t hi0 = smem_u32(tiles + s * kYStageBytes);
#pragma unroll
          for (int k = 0; k < KT / 8; k++) {
            const uint64_t a0 = desc_kmajor_sw128(hi0 + k * 32);                   // hi0; rows 0..255: hi0 | hi1
            const uint64_t a1 = desc_kmajor_sw128(hi0 + kTileBytes + k * 32);      // hi1
            const uint64_t b2 = desc_kmajor_sw128(hi0 + 2 * kTileBytes + k * 32);  // rows 0..255: 2 lo0 | 2 lo1
            mma_tf32(tmem_base, a0, a0, acc, kIdesc);
            mma_tf32(tmem_base, a0, b2, 1u, kIdesc);
            mma_tf32(tmem_base + 256, a1, a0, acc, kIdesc);
            mma_tf32(tmem_base + 256, a1, b2, 1u, kIdesc);
            acc = 1;
          }
          commit(&empty[s]);
          if (base + KT >= je) commit(accfull);
        }
        __syncwarp();
      }
      jc++;
    }
  } else {
    // ================================ EPILOGUE ================================
    // thread = accumulator lane: rows ew * 32 + lane of D_top and of D_bot, W = D / 2
    const int ew = warp - kYProducerWarps;
    const int row = ew * 32 + lane;
    unsigned long long jc = 0;
    for (long long j = blockIdx.x; j < a.n_jobs; j += gridDim.x) {
      float *out = a.W + (size_t)j * KY * KY;
      if (a.job_end[j] <= a.job_begin[j]) {
#pragma unroll 1
        for (int hb = 0; hb < 2; hb++) {
          float *o = out + (size_t)(hb * KP + row) * KY;
#pragma unroll 4
          for (int c = 0; c < KY; c += 4) *reinterpret_cast<float4 *>(o + c) = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        continue;
      }
      mbar_wait(accfull, (uint32_t)(jc & 1));
      fence_after();
#pragma unroll 1
      for (int hb = 0; hb < 2; hb++) {
        const uint32_t t0 = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(hb * 256);
        float *o = out + (size_t)(hb * KP + row) * KY;
#pragma unroll 1
        for (int c = 0; c < KY; c += 32) {
          uint32_t x[32];
          tmem_ld32(t0 + c, x);
          tmem_ld_wait();
#pragma unroll
          for (int q = 0; q < 32; q += 4)
            __stcs(reinterpret_cast<float4 *>(o + c + q),
                   make_float4(0.5f * __uint_as_float(x[q + 0]), 0.5f * __uint_as_float(x[q + 1]),
                               0.5f * __uint_as_float(x[q + 2]), 0.5f * __uint_as_float(x[q + 3])));
        }
      }
      fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(accempty);
      jc++;
    }
  }
  fence_before();
  __syncthreads();
  if (warp == kMmaWarp) tmem_dealloc(tmem_base, kTmemCols);
}


// G = scale * sum_j (W_j + W_j^T) over a contiguous run of partials (K1 finalize).
__global__ void wgram_reduce_sym_kernel(const float *__restrict__ W, int n_parts, float scale,
                                        float *__restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= KP * KP) return;
  const int r = i / KP, c = i % KP;
  float acc = 0.f;
  for (int p = 0; p < n_parts; p++) {
    const float *w = W + (size_t)p * KP * KP;
    acc += w[r * KP + c] + w[c * KP + r];
  }
  out[i] = scale * acc;
}

// Contiguous row blocks (multiples of KT rows) for the plain Gram.
__global__ void block_jobs_kernel(int64_t begin, int64_t end, int n_jobs, int64_t *jb, int64_t *je) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n_jobs) return;
  const int64_t n = end - begin;
  int64_t per = (n + n_jobs - 1) / n_jobs;
  per = (per + KT - 1) / KT * KT;
  const int64_t b = min(begin + (int64_t)j * per, end);
  jb[j] = b;
  je[j] = min(b + per, end);
}


constexpr size_t kSmemPlain = (size_t)STAGES * kStageBytes + 1024 + 12 * 8 + 16;

unsigned grid_for(int64_t n_jobs) {
  int dev = 0, sms = kNumSMsB200;
  CUDA_CHECK(cudaGetDevice(&dev));
  CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  return (unsigned)std::min<int64_t>(n_jobs, sms);
}

}  // namespace

void GramWorkspace::alloc(int jobs) {
  max_jobs = jobs;
  job_begin.alloc(jobs);
  job_end.alloc(jobs);
  W.alloc((size_t)jobs * KP * KP);
}

void launch_gram_tc(const float *Y, int64_t row_begin, int64_t row_end, float alpha0,
                    const GramWorkspace &ws, float *P, cudaStream_t s) {
  const int64_t n = row_end - row_begin;
  if (n <= 0) {
    CUDA_CHECK(cudaMemsetAsync(P, 0, sizeof(float) * KP * KP, s));
    return;
  }
  // at least 8 stages of work per job, at most one job per workspace slot
  const int n_jobs = (int)std::max<int64_t>(1, std::min<int64_t>(ws.max_jobs, n / (8 * KT)));
  block_jobs_kernel<<<1, 256, 0, s>>>(row_begin, row_end, n_jobs, ws.job_begin.get(), ws.job_end.get());
  count_launch();
  WGramArgs a{};
  a.Y = Y;
  a.ld = KP;
  a.job_begin = ws.job_begin.get();
  a.job_end = ws.job_end.get();
  a.n_jobs = n_jobs;
  a.W = ws.W.get();
  launch_wgram(a, s);
  launch_wgram_reduce_sym(ws.W.get(), n_jobs, alpha0, P, s);
}

// One 128 x 128 block per job.  a.Y may point into a wider row (Y + 128 with a.ld = 256: the
// second diagonal block of a 256-column Gram); a.ld is the true row stride.
void launch_wgram(const WGramArgs &a, cudaStream_t s) {
  if (a.n_jobs <= 0) return;
  if (a.ld < KP || a.ld % 4 != 0) throw NotImplemented("tensor-core Gram: the row stride must be >= 128");
  static PerDeviceOnce configured;
  configured.run([&] {
    CUDA_CHECK(cudaFuncSetAttribute(wgram_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemPlain));
  });
  wgram_kernel<<<grid_for(a.n_jobs), kThreads, kSmemPlain, s>>>(a);
  count_launch();
  CUDA_CHECK(cudaGetLastError());
}

// Whole 256 x 256 Gram of rows with stride a.ld >= 256: a.W receives W [256][256] per job
// (G = W + W^T), a.bpart (optional) kWGram256BParts x 256 partial sums of (bias + w) y per job.
void launch_wgram256(const WGramArgs &a, cudaStream_t s) {
  if (a.n_jobs <= 0) return;
  if (a.ld < KY || a.ld % 4 != 0) throw InvalidArgument("256-column Gram: row stride must be >= 256");
  constexpr size_t smem = (size_t)YSTAGES * kYStageBytes + 1024 + 128;
  static_assert(smem <= 232448, "256-column Gram stages do not fit shared memory");
  static PerDeviceOnce configured;
  configured.run([&] {
    CUDA_CHECK(cudaFuncSetAttribute(wgram256_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  });
  wgram256_kernel<<<grid_for(a.n_jobs), kYThreads, smem, s>>>(a);
  count_launch();
  CUDA_CHECK(cudaGetLastError());
}

void launch_wgram_reduce_sym(const float *W, int n_parts, float scale, float *out, cudaStream_t s) {
  wgram_reduce_sym_kernel<<<(KP * KP + 255) / 256, 256, 0, s>>>(W, n_parts, scale, out);
  count_launch();
  CUDA_CHECK(cudaGetLastError());
}

}  // namespace ials
