// K4 + K6 + K5 fused on the 5th-generation tensor cores: for a block of users,
//     S = user[b:e] item^T  ->  S[seen] = -inf  ->  first k of (-S, index)
// without the score matrix ever leaving the SM.  Replaces, as one kernel,
//   IALSTrainer::user_scores        /root/reference/cpp_source/als/IALSTrainer.hpp:942-984
//   the seen-item mask              /root/reference/src/irspack/evaluation/evaluator.py:426-432
//   the (-score, index) partial sort /root/reference/cpp_source/evaluator.cpp:324-355
//
// float32 parity on TF32 tensor cores (3xTF32): every operand is split into hi = tf32(x) and
// lo = x - hi (exact), and  x.y = hi.hi + hi.lo + lo.hi + O(2^-22 |x||y|).  Per k-step of 8
// features one N = 256 MMA  A_hi x [B_hi | B_lo]  puts hi.hi into accumulator columns 0-127 and
// hi.lo into 128-255, and one N = 128 MMA  A_lo x B_hi  adds lo.hi to columns 128-255; the
// epilogue adds the large and the small accumulator in fp32.
//
// One CTA = 128 users x one contiguous range of 128-item tiles (grid.y splits the catalogue when
// there are fewer user tiles than SMs).  416 threads, warp-specialised:
//   all warps   prologue: the user tile (128 x ld floats) is split and parked in shared memory
//               for the whole kernel, K-major SWIZZLE_128B, one 32-feature chunk per 32 KB.
//   warps 0-3   producers: a stage is one 32-feature chunk of 128 item rows (128-byte segments,
//               8 lanes per row), split into hi | lo tiles; the loads of the next stage are in
//               flight while the current one is converted.  3 stages x 32 KB.
//   warps 4-11  epilogue, thread = (user row = TMEM lane, column half of the tile): tcgen05.ld 16
//               columns at a time (the next 16 in flight), add, compare with the row's running
//               threshold tau (the score of its current k-th best); survivors that are not in
//               the row's mask are appended, as 64-bit keys (order-preserving(-score) << 32 |
//               index), to the thread's candidate buffer in global memory -- each thread on its
//               own, no warp vote per column.  A buffer that could not take another chunk is
//               compacted by the whole warp (bitonic sort across the lanes), which also tightens
//               tau.  The mask is a cursor into the row's sorted CSR column list with a four-deep
//               look-ahead queue in registers.
//   warp 12     MMA issuer (one lane) + TMEM owner; accumulators double-buffered (2 x 256 cols).
// A small second kernel merges the per-split candidate lists and writes (index, score, count).
#include <cub/block/block_radix_sort.cuh>

#include <climits>
#include <cstdlib>
#include <string>

#include "common.cuh"
#include "tc.cuh"

namespace ials {
namespace {

using namespace tc;

constexpr int TM = 128;      // users per CTA = UMMA M
constexpr int TN = 128;      // items per tile
constexpr int KC = 32;       // features per stage: one 128-byte swizzle row
constexpr int STAGES = 3;
constexpr int kMaxKc = 4;    // ld <= 128
constexpr int kTileBytes = TM * 128;         // 16 KB: 128 rows x 32 tf32
constexpr int kStageBytes = 2 * kTileBytes;  // hi | lo
constexpr int kProdWarps = 4, kProdGroup = 4;  // one group: every stage
constexpr int kEpiWarps = 8;                   // two per TMEM lane quadrant, 64 columns of a tile each
constexpr int kMmaWarp = kProdWarps + kEpiWarps;
constexpr int kThreads = (kProdWarps + kEpiWarps + 1) * kWarp;  // 416
constexpr int kTmemCols = 512;
static_assert(kProdWarps % 4 == 0, "epilogue warps must start on a TMEM lane quadrant");

constexpr uint32_t kIdescN256 = idesc_tf32(TM, 256, false, false);
constexpr uint32_t kIdescN128 = idesc_tf32(TM, 128, false, false);

struct ScoreTcArgs {
  const float *users;  // first row of the user block [n_rows x ld]
  int64_t n_rows;
  const float *items;  // [n_items x ld]
  int64_t n_items;
  int ld;
  // mask: CSR whose row (m_row0 + r) lists, strictly ascending, the items hidden from block row r
  const int64_t *m_indptr;
  const int32_t *m_indices;
  const float *m_data;  // optional: stored zeros do not mask (scipy's .nonzero())
  int64_t m_row0;
  const int64_t *m_rowmap;  // optional: block row r is masked by CSR row m_row0 + m_rowmap[r]
  // allow-lists (recommendable items, evaluator.py:115-136 / util.hpp:426-504): CSR whose row lists,
  // strictly ascending, the ONLY items block row r may receive (row a_row0 + r).  a_n_lists 0: none;
  // 1: one list shared by every row, given as a bitmap instead (bit i & 31 of word i >> 5 = item i
  // is allowed; one cached word per 16-column chunk replaces a walk over the whole list per row)
  const int64_t *a_indptr;
  const int32_t *a_indices;
  const uint32_t *a_bitmap;
  int64_t a_row0;
  int a_n_lists;
  int k;
  int n_splits, tiles_per_split;
  unsigned long long *cand;  // [n_rows][n_splits][32 * M] candidate keys
  float *out_scores;         // dense mode: [n_rows x out_ld], no mask / top-k
  int64_t out_ld;
};

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
__device__ __forceinline__ unsigned long long shfl_xor_u64(unsigned long long v, int m) {
  return __shfl_xor_sync(0xffffffffu, v, m);
}

// Ascending bitonic sort of 32 * M keys held M per lane (element e = lane * M + i).
template <int M>
__device__ __forceinline__ void warp_sort(unsigned long long (&v)[M], int lane) {
#pragma unroll
  for (int k2 = 2; k2 <= 32 * M; k2 <<= 1) {
#pragma unroll
    for (int j = k2 >> 1; j > 0; j >>= 1) {
      if (j >= M) {
        const int lm = j / M;
#pragma unroll
        for (int i = 0; i < M; i++) {
          const unsigned long long o = shfl_xor_u64(v[i], lm);
          const bool up = (((lane * M + i) & k2) == 0), lower = (lane & lm) == 0;
          const unsigned long long mn = v[i] < o ? v[i] : o, mx = v[i] < o ? o : v[i];
          v[i] = (lower == up) ? mn : mx;
        }
      } else {
#pragma unroll
        for (int i = 0; i < M; i++) {
          if ((i & j) == 0) {
            const unsigned long long x = v[i], y = v[i | j];
            const bool up = (((lane * M + i) & k2) == 0);
            const bool sw = (x > y) == up;
            v[i] = sw ? y : x;
            v[i | j] = sw ? x : y;
          }
        }
      }
    }
  }
}

// The whole warp compacts the candidate buffer of lane `src`'s row: sort its first n keys,
// keep the best k at the front (padded with ~0).  Returns the new threshold of that row
// (score of its k-th best; -inf while it has fewer than k candidates).
template <int M>
__device__ __noinline__ float compact_row(unsigned long long *buf, int n, int k, int lane) {
  unsigned long long v[M];
#pragma unroll
  for (int i = 0; i < M; i++) {
    const int e = lane * M + i;
    v[i] = e < n ? __ldcg(buf + e) : ~0ull;
  }
  warp_sort<M>(v, lane);
  unsigned long long kth = ~0ull;
#pragma unroll
  for (int i = 0; i < M; i++) {
    const int e = lane * M + i;
    if (e < k) __stcg(buf + e, v[i]);
    if (e == k - 1) kth = v[i];
  }
  kth = __shfl_sync(0xffffffffu, kth, (k - 1) / M);
  __syncwarp();
  return (n >= k && kth != ~0ull) ? key_score(kth) : -INFINITY;
}

__device__ __forceinline__ float4 tf32_hi(float4 u) {
  return make_float4(__uint_as_float(__float_as_uint(u.x) & 0xffffe000u),
                     __uint_as_float(__float_as_uint(u.y) & 0xffffe000u),
                     __uint_as_float(__float_as_uint(u.z) & 0xffffe000u),
                     __uint_as_float(__float_as_uint(u.w) & 0xffffe000u));
}
__device__ __forceinline__ float4 sub4(float4 a, float4 b) {
  return make_float4(a.x - b.x, a.y - b.y, a.z - b.z, a.w - b.w);
}

// ALLOW: the allow-list cursor is compiled in (a separate instantiation: without it the kernel
// keeps the register budget it was tuned to)
template <int M, bool ALLOW>
__global__ void __launch_bounds__(kThreads, 1) score_tc_kernel(ScoreTcArgs a) {
  constexpr int CAP = 32 * M;
  extern __shared__ unsigned char smem_raw[];
  // dynamic shared memory is only guaranteed 16-byte aligned: round up to the swizzle atom
  unsigned char *base = reinterpret_cast<unsigned char *>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  unsigned char *As = base;                          // [kMaxKc][hi 16 KB | lo 16 KB]
  unsigned char *Bs = base + kMaxKc * kStageBytes;   // [STAGES][hi | lo]
  uint64_t *bars = reinterpret_cast<uint64_t *>(Bs + STAGES * kStageBytes);
  uint64_t *full = bars;                      // [STAGES] producers -> MMA
  uint64_t *empty = bars + STAGES;            // [STAGES] MMA (commit) -> producers
  uint64_t *accfull = bars + 2 * STAGES;      // [2] MMA (commit) -> epilogue
  uint64_t *accempty = accfull + 2;           // [2] epilogue -> MMA
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(accempty + 2);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int ld = a.ld, n_kc = ld / KC;
  const int64_t row0 = (int64_t)blockIdx.x * TM;
  const int split = (int)blockIdx.y;
  const int tiles_total = (int)((a.n_items + TN - 1) / TN);
  const int tile_begin = split * a.tiles_per_split;
  const int n_tiles = min(a.tiles_per_split, tiles_total - tile_begin);

  if (tid == 0) {
    for (int s = 0; s < STAGES; s++) {
      mbar_init(&full[s], kProdGroup);
      mbar_init(&empty[s], 1);
    }
    for (int b = 0; b < 2; b++) {
      mbar_init(&accfull[b], 1);
      mbar_init(&accempty[b], kEpiWarps);
    }
    mbar_init_fence();
  }
  if (warp == kMmaWarp) tmem_alloc(tmem_slot, kTmemCols);

  // ---- prologue: the user tile, split and swizzled, stays in shared memory ----
  {
    const int f4_per_row = ld / 4;
    for (int f = tid; f < TM * f4_per_row; f += kThreads) {
      const int r = f / f4_per_row, c = f % f4_per_row;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (row0 + r < a.n_rows) v = __ldg(reinterpret_cast<const float4 *>(a.users + (row0 + r) * ld + 4 * c));
      const float4 h = tf32_hi(v), l = sub4(v, h);
      unsigned char *dst = As + (c >> 3) * kStageBytes + sw128_offset(r, c & 7);
      *reinterpret_cast<float4 *>(dst) = h;
      *reinterpret_cast<float4 *>(dst + kTileBytes) = l;
    }
    fence_proxy_async_smem();
  }
  fence_before();
  __syncthreads();
  fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < kProdWarps) {
    // ================================ PRODUCERS ================================
    // One group serves every stage, so its loop is kept lean (r02o: 348 instructions per stage
    // and warp made the producers the bottleneck of the eight-warp epilogue): the lane's eight
    // row pointers advance by constants, the stage index and its phase are counters, only the
    // last tile of the catalogue checks its rows, and the two register buffers swap roles in a
    // loop unrolled by two instead of being copied.
    const int pw = warp;
    const int rsub = lane >> 3, c16 = lane & 7;
    const unsigned total = (unsigned)n_tiles * (unsigned)n_kc;
    uint32_t offs[8];  // swizzled byte offsets of this lane's eight 16-byte chunks in a tile
#pragma unroll
    for (int i = 0; i < 8; i++) offs[i] = sw128_offset(32 * pw + 4 * i + rsub, c16);
    const size_t row_step = (size_t)4 * ld;  // the lane's rows are 4 apart
    // cursor of the NEXT load: tile, feature chunk, pointer to this lane's first row
    int lt = 0, lkc = 0;
    const float *lsrc = a.items + ((size_t)tile_begin * TN + 32 * pw + rsub) * ld + c16 * 4;
    auto load = [&](float4(&v)[8]) {
      const int64_t j0 = (int64_t)(tile_begin + lt) * TN + 32 * pw + rsub;
      if (j0 + 28 < a.n_items) {  // every row of this lane exists (all tiles but the last)
#pragma unroll
        for (int i = 0; i < 8; i++) v[i] = __ldg(reinterpret_cast<const float4 *>(lsrc + i * row_step));
      } else {
#pragma unroll
        for (int i = 0; i < 8; i++)
          v[i] = j0 + 4 * i < a.n_items ? __ldg(reinterpret_cast<const float4 *>(lsrc + i * row_step))
                                        : make_float4(0.f, 0.f, 0.f, 0.f);
      }
      lsrc += KC;
      if (++lkc == n_kc) {
        lkc = 0;
        lt++;
        lsrc += (size_t)TN * ld - (size_t)n_kc * KC;
      }
    };
    int s = 0;
    uint32_t ph = 1;  // parity to wait for on empty[s]: the first pass over the ring is free
    auto convert = [&](const float4(&v)[8]) {
      mbar_wait(&empty[s], ph);
      unsigned char *hi = Bs + s * kStageBytes;
#pragma unroll
      for (int i = 0; i < 8; i++) {
        const float4 h = tf32_hi(v[i]), l = sub4(v[i], h);
        *reinterpret_cast<float4 *>(hi + offs[i]) = h;
        *reinterpret_cast<float4 *>(hi + kTileBytes + offs[i]) = l;
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&full[s]);
      if (++s == STAGES) {
        s = 0;
        ph ^= 1;
      }
    };
    float4 va[8], vb[8];
    if (total > 0) load(va);
    for (unsigned it = 0; it < total; it += 2) {
      if (it + 1 < total) load(vb);
      convert(va);
      if (it + 1 < total) {
        if (it + 2 < total) load(va);
        convert(vb);
      }
    }
  } else if (warp == kMmaWarp) {
    // ================================ MMA ISSUER ================================
    unsigned it = 0;
    for (int t = 0; t < n_tiles; t++) {
      const int buf = t & 1;
      mbar_wait(&accempty[buf], (uint32_t)(((t >> 1) & 1) ^ 1));
      fence_after();
      const uint32_t d = tmem_base + (uint32_t)(buf * 256);
      for (int kc = 0; kc < n_kc; kc++, it++) {
        const int s = (int)(it % STAGES);
        mbar_wait(&full[s], (it / STAGES) & 1);
        fence_after();
        if (lane == 0) {
          const uint32_t a_hi = smem_u32(As + kc * kStageBytes), a_lo = a_hi + kTileBytes;
          const uint32_t b = smem_u32(Bs + s * kStageBytes);
#pragma unroll
          for (int kk = 0; kk < KC / 8; kk++) {
            const uint64_t db = desc_kmajor_sw128(b + kk * 32);
            mma_tf32(d, desc_kmajor_sw128(a_hi + kk * 32), db, (kc | kk) != 0, kIdescN256);
            mma_tf32(d + 128, desc_kmajor_sw128(a_lo + kk * 32), db, 1u, kIdescN128);
          }
          commit(&empty[s]);
          if (kc == n_kc - 1) commit(&accfull[buf]);
        }
        __syncwarp();
      }
    }
  } else {
    // ================================ EPILOGUE ================================
    // Eight warps (r02l: with four, the epilogue took 9.3 k cycles per tile against 3.3 k of
    // tensor time): warp = (TMEM lane quadrant, column half).  The two threads of a row keep
    // separate candidate lists -- one more list per row and split for the merge kernel.
    const int q = warp & 3;               // TMEM lane quadrant of this warp
    const int half = (warp - kProdWarps) >> 2;
    const int cbeg = (TN / 2) * half;     // this warp's columns of every tile: [cbeg, cbeg + 64)
    const int64_t rb = row0 + q * 32 + lane;  // row of the user block owned by this thread
    const bool row_ok = rb < a.n_rows;
    const bool dense = a.out_scores != nullptr;
    unsigned long long *buf_row =
        dense ? nullptr : a.cand + (((size_t)(row_ok ? rb : 0) * a.n_splits + split) * 2 + half) * CAP;
    int count = 0;
    float tau = -INFINITY;
    // mask cursor (strictly ascending column ids) with a four-deep look-ahead queue: the next
    // four (column, stored value) pairs of the row sit in registers, so advancing the cursor
    // never waits for the load it issues (ncu r02e: one exposed global-load latency per warp
    // and 32-column chunk, every chunk -- some lane of the 32 rows always had a seen item)
    int64_t mp = 0, me = 0;
    int n0 = INT_MAX, n1 = INT_MAX, n2 = INT_MAX, n3 = INT_MAX;
    float z0 = 1.f, z1 = 1.f, z2 = 1.f, z3 = 1.f;
    if (row_ok && !dense && a.m_indptr != nullptr) {
      const int64_t mr = a.m_row0 + (a.m_rowmap ? a.m_rowmap[rb] : rb);
      mp = a.m_indptr[mr];
      me = a.m_indptr[mr + 1];
      const int first_col = tile_begin * TN;
      int64_t lo = mp, hi = me;  // lower bound of first_col
      while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (a.m_indices[mid] < first_col) lo = mid + 1; else hi = mid;
      }
      mp = lo;
      if (mp < me) { n0 = a.m_indices[mp]; if (a.m_data) z0 = a.m_data[mp]; }
      if (mp + 1 < me) { n1 = a.m_indices[mp + 1]; if (a.m_data) z1 = a.m_data[mp + 1]; }
      if (mp + 2 < me) { n2 = a.m_indices[mp + 2]; if (a.m_data) z2 = a.m_data[mp + 2]; }
      if (mp + 3 < me) { n3 = a.m_indices[mp + 3]; if (a.m_data) z3 = a.m_data[mp + 3]; }
    }
    // allow-list cursor (two-deep look-ahead)
    const bool allow = ALLOW && !dense && a.a_n_lists > 0;
    int64_t ap = 0, ae = 0;
    int q0 = INT_MAX, q1 = INT_MAX;
    if (ALLOW && row_ok && allow && a.a_n_lists != 1) {
      const int64_t ar = a.a_row0 + rb;
      ap = a.a_indptr[ar];
      ae = a.a_indptr[ar + 1];
      const int first_col = tile_begin * TN;
      int64_t lo = ap, hi = ae;
      while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (a.a_indices[mid] < first_col) lo = mid + 1; else hi = mid;
      }
      ap = lo;
      if (ap < ae) q0 = a.a_indices[ap];
      if (ap + 1 < ae) q1 = a.a_indices[ap + 1];
    }
    const int k = a.k;

    for (int t = 0; t < n_tiles; t++) {
      const int buf = t & 1;
      mbar_wait(&accfull[buf], (uint32_t)((t >> 1) & 1));
      fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * 256);
      const int64_t c0 = (int64_t)(tile_begin + t) * TN;
      const int ncols = (int)min((int64_t)TN, a.n_items - c0);
      // 16 columns per chunk (a 13-warp CTA gets 128 registers per thread: registers are handed
      // out to groups of four warps; 32-column chunks with their prefetch spilled in this loop,
      // r02k); the accumulator columns of chunk c + CH travel from TMEM while chunk c is examined
      constexpr int CH = 16;
      uint32_t big[CH], sml[CH];
      tmem_ld16(taddr + cbeg, big);
      tmem_ld16(taddr + 128 + cbeg, sml);
#pragma unroll 1
      for (int c = cbeg; c < cbeg + TN / 2; c += CH) {
        if (c >= ncols) break;  // warp-uniform
        tmem_ld_wait();
        float sc[CH];
#pragma unroll
        for (int e = 0; e < CH; e++) sc[e] = __uint_as_float(big[e]) + __uint_as_float(sml[e]);
        if (c + CH < ncols && c + CH < cbeg + TN / 2) {
          tmem_ld16(taddr + c + CH, big);
          tmem_ld16(taddr + 128 + c + CH, sml);
        }
        const int jbase = (int)c0 + c;
        if (dense) {
          if (row_ok) {
            float *dst = a.out_scores + rb * a.out_ld + jbase;
            if ((a.out_ld & 3) == 0 && c + CH <= ncols) {
#pragma unroll
              for (int e = 0; e < CH; e += 4)
                *reinterpret_cast<float4 *>(dst + e) = make_float4(sc[e], sc[e + 1], sc[e + 2], sc[e + 3]);
            } else {
#pragma unroll
              for (int e = 0; e < CH; e++)
                if (c + e < ncols) dst[e] = sc[e];
            }
          }
          continue;
        }
        // columns of this chunk hidden by the mask (bit e = column jbase + e)
        uint32_t mbits = 0;
        while (n0 < jbase + CH) {  // divergent; the queue keeps it free of load latency
          if (n0 >= jbase && z0 != 0.f) mbits |= 1u << (n0 - jbase);  // stored zeros do not mask
          n0 = n1; z0 = z1;
          n1 = n2; z1 = z2;
          n2 = n3; z2 = z3;
          mp++;
          const bool more = mp + 3 < me;
          n3 = more ? a.m_indices[mp + 3] : INT_MAX;
          z3 = (more && a.m_data) ? a.m_data[mp + 3] : 1.f;
        }
        if (ALLOW && allow) {  // everything outside the row's allow-list is hidden as well
          uint32_t abits = 0;
          if (a.a_n_lists == 1) {  // jbase is a multiple of CH: the chunk lies inside one word
            static_assert(32 % CH == 0 && TN % CH == 0, "a chunk must not straddle bitmap words");
            abits = (a.a_bitmap[jbase >> 5] >> (jbase & 31)) & ((1u << CH) - 1u);
          } else {
            while (q0 < jbase + CH) {
              if (q0 >= jbase) abits |= 1u << (q0 - jbase);
              q0 = q1;
              ap++;
              q1 = ap + 1 < ae ? a.a_indices[ap + 1] : INT_MAX;
            }
          }
          mbits |= ~abits;
        }
        if (c + CH > ncols) mbits |= ~0u << (ncols - c);  // columns past the catalogue
        if (!row_ok) mbits = ~0u;
        // Thread = row: every lane decides for its own row, without a warp vote per column
        // (r02e: 32 dependent votes per chunk set the pace of the kernel, the tensor pipe ran at
        // 16 %).  A row appends what beats its threshold; the candidate buffer always has room
        // for one chunk, the warp-wide compaction runs between chunks.
        uint32_t hb = 0;
#pragma unroll
        for (int e = 0; e < CH; e++) hb |= sc[e] > tau ? (1u << e) : 0u;
        hb &= ~mbits;
        // one trip per hit of the lane with the most hits (usually one): the column's score is
        // picked from the registers by a select tree instead of CH predicated append blocks
        while (hb != 0) {
          const int e = __ffs(hb) - 1;
          hb &= hb - 1;
          float m8[8], m4[4];
#pragma unroll
          for (int i = 0; i < 8; i++) m8[i] = (e & 8) ? sc[8 + i] : sc[i];
#pragma unroll
          for (int i = 0; i < 4; i++) m4[i] = (e & 4) ? m8[4 + i] : m8[i];
          const float a0 = (e & 2) ? m4[2] : m4[0], a1 = (e & 2) ? m4[3] : m4[1];
          const float s = (e & 1) ? a1 : a0;
          __stcg(buf_row + count, make_key(s, (uint32_t)(jbase + e)));
          count++;
        }
        unsigned fullm = __ballot_sync(0xffffffffu, count > CAP - CH);
        if (fullm) {
          while (fullm) {
            const int src = __ffs(fullm) - 1;
            fullm &= fullm - 1;
            unsigned long long *b = reinterpret_cast<unsigned long long *>(
                __shfl_sync(0xffffffffu, (unsigned long long)buf_row, src));
            const int n = __shfl_sync(0xffffffffu, count, src);
            __syncwarp();
            const float nt = compact_row<M>(b, n, k, lane);
            if (lane == src) {
              tau = nt;
              count = k;
            }
          }
          // the prefetched columns are fetched again instead of being kept alive across the calls
          if (c + CH < ncols && c + CH < cbeg + TN / 2) {
            tmem_ld_wait();
            tmem_ld16(taddr + c + CH, big);
            tmem_ld16(taddr + 128 + c + CH, sml);
          }
        }
      }
      tmem_ld_wait();  // (a prefetch issued for a tile that ends before this warp's columns)
      fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&accempty[buf]);
    }
    if (!dense) {
      // final compaction of every row of this warp: sorted best k at the front, ~0 padding
      for (int src = 0; src < 32; src++) {
        const int n = __shfl_sync(0xffffffffu, count, src);
        const bool ok = __shfl_sync(0xffffffffu, (int)row_ok, src) != 0;
        unsigned long long *b = reinterpret_cast<unsigned long long *>(
            __shfl_sync(0xffffffffu, (unsigned long long)buf_row, src));
        if (!ok) continue;  // warp-uniform
        __syncwarp();
        compact_row<M>(b, n, k, lane);
      }
    }
  }

  // teardown: everybody done with TMEM before the owner frees it
  fence_before();
  __syncthreads();
  if (warp == kMmaWarp) tmem_dealloc(tmem_base, kTmemCols);
}

// Merge the per-split sorted candidate lists of a row: first k of the union.
constexpr int kMgThreads = 256, kMgItems = 8, kMgCap = kMgThreads * kMgItems;
__global__ void __launch_bounds__(kMgThreads)
merge_topk_kernel(const unsigned long long *__restrict__ cand, int64_t n_rows, int n_splits, int cap,
                  int k, int32_t *__restrict__ out_idx, float *__restrict__ out_score,
                  int32_t *__restrict__ out_count) {
  using Sort = cub::BlockRadixSort<unsigned long long, kMgThreads, kMgItems>;
  __shared__ typename Sort::TempStorage tmp;
  __shared__ unsigned long long sorted[kMgCap];
  const int tid = threadIdx.x;
  for (int64_t row = blockIdx.x; row < n_rows; row += gridDim.x) {
    const unsigned long long *src = cand + (size_t)row * n_splits * cap;
    if (n_splits == 1) {  // already sorted by the producer of the list
      for (int i = tid; i < k; i += kMgThreads) sorted[i] = src[i];
      __syncthreads();
    } else if (n_splits <= 4) {
      // a few sorted lists of distinct keys (the column is part of the key): an element's place
      // in the union is its own position plus the number of smaller keys in the other lists
      for (int i = tid; i < k; i += kMgThreads) sorted[i] = ~0ull;
      __syncthreads();
      for (int e = tid; e < n_splits * k; e += kMgThreads) {
        const int l = e / k, i = e - l * k;
        const unsigned long long key = src[(size_t)l * cap + i];
        if (key == ~0ull) continue;
        int pos = i;
        for (int l2 = 0; l2 < n_splits; l2++) {
          if (l2 == l) continue;
          const unsigned long long *o = src + (size_t)l2 * cap;
          int lo = 0, hi = k;  // first index whose key is not smaller (~0 padding sorts last)
          while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (o[mid] < key) lo = mid + 1; else hi = mid;
          }
          pos += lo;
        }
        if (pos < k) sorted[pos] = key;
      }
      __syncthreads();
    } else {
      unsigned long long keys[kMgItems];
#pragma unroll
      for (int i = 0; i < kMgItems; i++) {
        const int p = tid * kMgItems + i;
        keys[i] = p < n_splits * k ? src[(size_t)(p / k) * cap + (p % k)] : ~0ull;
      }
      Sort(tmp).Sort(keys);
      __syncthreads();
#pragma unroll
      for (int i = 0; i < kMgItems; i++) sorted[tid * kMgItems + i] = keys[i];
      __syncthreads();
    }
    __shared__ int cnt;
    if (tid == 0) cnt = 0;
    __syncthreads();
    int mine = 0;
    for (int i = tid; i < k; i += kMgThreads) {
      const unsigned long long key = sorted[i];
      const bool ok = key != ~0ull;
      out_idx[row * k + i] = ok ? (int32_t)(key & 0xffffffffu) : -1;
      if (out_score) out_score[row * k + i] = ok ? key_score(key) : -INFINITY;
      mine += ok ? 1 : 0;
    }
    if (mine) atomicAdd(&cnt, mine);
    __syncthreads();
    if (tid == 0) out_count[row] = cnt;
    __syncthreads();
  }
}

__global__ void csr_sorted_kernel(const int64_t *__restrict__ indptr, const int32_t *__restrict__ indices,
                                  int64_t n_rows, int *__restrict__ unsorted) {
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / kWarp;
  const int lane = threadIdx.x % kWarp;
  if (warp >= n_rows) return;
  const int64_t s = indptr[warp], e = indptr[warp + 1];
  bool bad = false;
  for (int64_t j = s + 1 + lane; j < e; j += kWarp) bad |= indices[j - 1] >= indices[j];
  if (bad) atomicExch(unsorted, 1);
}

template <int M, bool ALLOW>
void launch_fused_as(const ScoreTcArgs &a, int user_tiles, cudaStream_t s) {
  const size_t smem = (size_t)(kMaxKc + STAGES) * kStageBytes + 1024 + 16 * 8;
  static PerDeviceOnce configured;
  configured.run([&] {
    CUDA_CHECK(cudaFuncSetAttribute(score_tc_kernel<M, ALLOW>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)smem));
  });
  dim3 grid((unsigned)user_tiles, (unsigned)a.n_splits);
  score_tc_kernel<M, ALLOW><<<grid, kThreads, smem, s>>>(a);
  count_launch();
  CUDA_CHECK(cudaGetLastError());
}
template <int M>
void launch_fused(const ScoreTcArgs &a, int user_tiles, cudaStream_t s) {
  if (a.a_n_lists > 0) launch_fused_as<M, true>(a, user_tiles, s);
  else launch_fused_as<M, false>(a, user_tiles, s);
}

}  // namespace

bool score_tc_supported(int ld, int64_t k) { return ld % 32 == 0 && ld >= 32 && ld <= 128 && k >= 1 && k <= 128; }
// candidate keys per row, split and column half: k + one 16-column chunk + room between two
// compactions (128 keys for k = 10 measured slower than 64: r02n 8.97 against r02l 8.43 ms)
int score_tc_capacity(int64_t k) { return k <= 16 ? 64 : (k <= 48 ? 128 : 256); }

// Catalogue splits for `n_rows` users: CTAs for (at most) two full waves, at least 4 item tiles each,
// and at most kMgCap keys per row in the merge.
int score_tc_splits(int64_t n_rows, int64_t n_items, int64_t k) {
  const int64_t user_tiles = ceil_div(n_rows, TM), tiles = ceil_div(n_items, TN);
  int64_t splits = std::max<int64_t>(1, (2 * kNumSMsB200) / user_tiles);  // at most two full waves of CTAs
  splits = std::min<int64_t>(splits, std::max<int64_t>(1, tiles / 4));
  splits = std::min<int64_t>(splits, std::max<int64_t>(1, kMgCap / (2 * k)));  // two lists per split
  splits = std::max<int64_t>(1, std::min<int64_t>(splits, 65535));
  const int64_t per = ceil_div(tiles, splits);
  return (int)ceil_div(tiles, per);
}
size_t score_tc_scratch_bytes(int64_t n_rows, int64_t n_items, int64_t k) {
  return sizeof(unsigned long long) * (size_t)n_rows * 2 * score_tc_splits(n_rows, n_items, k) * score_tc_capacity(k);
}

bool csr_rows_strictly_sorted(const int64_t *indptr, const int32_t *indices, int64_t n_rows,
                              cudaStream_t s) {
  if (n_rows == 0) return true;
  DeviceBuffer<int> d_flag;
  StreamSyncOnExit sync{s};
  d_flag.alloc(1);
  CUDA_CHECK(cudaMemsetAsync(d_flag.get(), 0, sizeof(int), s));
  const int T = 256;
  csr_sorted_kernel<<<(unsigned)ceil_div(n_rows * kWarp, T), T, 0, s>>>(indptr, indices, n_rows, d_flag.get());
  count_launch();
  CUDA_CHECK(cudaGetLastError());
  int h = 0;
  CUDA_CHECK(cudaMemcpyAsync(&h, d_flag.get(), sizeof(int), cudaMemcpyDeviceToHost, s));
  CUDA_CHECK(cudaStreamSynchronize(s));
  return h == 0;
}

// Fused scores + mask + top-k of a user block.  `scratch` holds score_tc_scratch_bytes().
void launch_score_topk_tc(const float *user_rows, int64_t n_rows, const float *item, int64_t n_items,
                          int ld, const int64_t *m_indptr, const int32_t *m_indices, const float *m_data,
                          int64_t m_row0, int k, void *scratch, int32_t *out_idx, float *out_score,
                          int32_t *out_count, cudaStream_t s, int a_n_lists, const int64_t *a_indptr,
                          const int32_t *a_indices, int64_t a_row0, const uint32_t *a_bitmap,
                          const int64_t *m_rowmap) {
  if (n_rows == 0) return;
  if (!score_tc_supported(ld, k)) throw NotImplemented("tensor-core top-k: ld must be 32..128 and k <= 128");
  if (n_items >= (1ll << 31) - 256) throw InvalidArgument("too many items");
  ScoreTcArgs a{};
  a.users = user_rows;
  a.n_rows = n_rows;
  a.items = item;
  a.n_items = n_items;
  a.ld = ld;
  a.m_indptr = m_indptr;
  a.m_indices = m_indices;
  a.m_data = m_data;
  a.m_row0 = m_row0;
  a.a_n_lists = a_n_lists;
  a.a_indptr = a_indptr;
  a.a_indices = a_indices;
  a.a_row0 = a_row0;
  a.a_bitmap = a_bitmap;
  a.m_rowmap = m_rowmap;
  if (a_n_lists == 1 && a_bitmap == nullptr) throw std::invalid_argument("shared allow-list needs its bitmap");
  a.k = k;
  a.n_splits = score_tc_splits(n_rows, n_items, k);
  a.tiles_per_split = (int)ceil_div(ceil_div(n_items, TN), a.n_splits);
  a.cand = static_cast<unsigned long long *>(scratch);
  const int user_tiles = (int)ceil_div(n_rows, TM);
  const int cap = score_tc_capacity(k);
  switch (cap) {
    case 64: launch_fused<2>(a, user_tiles, s); break;
    case 128: launch_fused<4>(a, user_tiles, s); break;
    default: launch_fused<8>(a, user_tiles, s); break;
  }
  const unsigned grid = (unsigned)std::min<int64_t>(n_rows, (int64_t)kNumSMsB200 * 8);
  merge_topk_kernel<<<grid, kMgThreads, 0, s>>>(a.cand, n_rows, 2 * a.n_splits, cap, k, out_idx, out_score,
                                                 out_count);
  count_launch();
  CUDA_CHECK(cudaGetLastError());
}

// Dense score block on the tensor cores (same arithmetic, scores written out).
void launch_scores_tc(const float *user_rows, int64_t n_rows, const float *item, int64_t n_items, int ld,
                      float *out, int64_t out_ld, cudaStream_t s) {
  if (n_rows == 0 || n_items == 0) return;
  if (!score_tc_supported(ld, 1)) throw NotImplemented("tensor-core scores: ld must be 32..128");
  ScoreTcArgs a{};
  a.users = user_rows;
  a.n_rows = n_rows;
  a.items = item;
  a.n_items = n_items;
  a.ld = ld;
  a.k = 1;
  a.n_splits = score_tc_splits(n_rows, n_items, 1);
  a.tiles_per_split = (int)ceil_div(ceil_div(n_items, TN), a.n_splits);
  a.out_scores = out;
  a.out_ld = out_ld;
  launch_fused<2>(a, (int)ceil_div(n_rows, TM), s);
}

}  // namespace ials
