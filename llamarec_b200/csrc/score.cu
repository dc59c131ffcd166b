// Host launchers for catalogue scoring (+ the exact-fp32 FFMA variant for small catalogues).
//   lrb_score_topk   precision 0 -> score_topk_tc_kernel (tcgen05/TMEM/TMA, bf16 operands)
//                    precision 1 -> score_topk_f32_kernel (fp32 FFMA, bit-comparable with the
//                                   fp32 reference `x @ E^T + bias`, model/lru.py:85)
//   lrb_score_dense  API-compatible dense logits for LRURec.forward
//   lrb_score_collect  bf16 tensor-core scores, every item at or above a per-user threshold collected
//                      (candidate pass of precision="exact", see exact.cu); lrb_score_collect_scores also
//                      stores the collected scores (candidate pass of the wide top-K)
//   lrb_wide_sample_threshold / lrb_wide_select  top-K lists of up to LRB_MAX_K_WIDE entries on the bf16 path
//                      (DESIGN.md section 2.2)
#include "api_util.h"
#include "score_topk_tc.cuh"

#include <cuda.h>
#include <climits>
#include <cmath>

namespace lrb {

constexpr double RESTART_TILES = 150.0;   // cost of one streaming top-K (re)start, in item tiles (see decompose())
constexpr int NS_PAIR = 4;                // TMA stages of the K <= 20 CTA-pair kernel (20 KB each)

// ============================================================================================
// fp32 path.  Thread = user row (state in registers), CTA = 128 rows, item chunks of 64 rows
// staged in shared memory and read with broadcast LDS.128.
// ============================================================================================
namespace f32 {

constexpr int ROWS = 128;   // users per CTA
constexpr int IT = 64;      // items per shared-memory chunk
constexpr int D = 64;

struct Params {
  const float* u;        // [B][64]
  const float* table;    // [rows][64]
  const float* bias_pad; // [ceil(rows/256)*256]
  int B;
  int rows;
  int row_offset;
  int K;
  const int* excl_sorted;
  const uint32_t* excl_bloom;
  int excl_stride;
  float* part_scores;
  int* part_ids;
  int* part_cnt;
  int slots;             // == number of item splits == gridDim.y
  float* dense_out;
  long long dense_ld;
};

template <bool kDense>
__global__ void __launch_bounds__(ROWS) score_f32_kernel(const Params p) {
  extern __shared__ __align__(16) uint8_t smem[];
  float* sE = reinterpret_cast<float*>(smem);                  // [IT][64]
  float* sBias = sE + IT * D;                                   // [IT]
  float* sOut = sBias + IT;                                     // dense: [ROWS][IT+1]
  float* sListS = sBias + IT;                                   // topk:  [K][ROWS]
  int* sListI = reinterpret_cast<int*>(sListS + (kDense ? 0 : p.K * ROWS));
  __shared__ int sCnt[2 * ROWS];   // [0..ROWS) entries held, [ROWS..2*ROWS) index of the worst entry

  const int tid = threadIdx.x;
  const int b = blockIdx.x * ROWS + tid;
  const bool live = b < p.B;

  float u[D];
#pragma unroll
  for (int k = 0; k < D; k += 4) {
    float4 v = live ? *reinterpret_cast<const float4*>(p.u + static_cast<size_t>(b) * D + k)
                    : make_float4(0.f, 0.f, 0.f, 0.f);
    u[k] = v.x; u[k + 1] = v.y; u[k + 2] = v.z; u[k + 3] = v.w;
  }

  // item range of this split, aligned to chunks
  const int chunks = (p.rows + IT - 1) / IT;
  const int c0 = static_cast<int>((static_cast<long long>(blockIdx.y) * chunks) / gridDim.y);
  const int c1 = static_cast<int>((static_cast<long long>(blockIdx.y + 1) * chunks) / gridDim.y);

  float own_thr = -INFINITY;
  const int* excl = nullptr;
  uint32_t bloom0 = 0u, bloom1 = 0u, bloom2 = 0u, bloom3 = 0u;
  if (!kDense) {
    sCnt[tid] = 0;
    if (live && p.excl_sorted != nullptr) {
      excl = p.excl_sorted + static_cast<size_t>(b) * p.excl_stride;
      const uint4 bw = *reinterpret_cast<const uint4*>(p.excl_bloom + static_cast<size_t>(b) * 4);
      bloom0 = bw.x; bloom1 = bw.y; bloom2 = bw.z; bloom3 = bw.w;
    }
  }
  const uint32_t ls_a = smem_u32(sListS + tid);
  const uint32_t li_a = smem_u32(sListI + tid);
  const uint32_t ln_a = smem_u32(&sCnt[tid]);
  const int limit_gid = p.row_offset + p.rows;

  for (int c = c0; c < c1; ++c) {
    const int i0 = c * IT;
    __syncthreads();
    // stage IT x 64 floats (zero beyond rows) and the bias
    for (int e = tid; e < IT * D / 4; e += ROWS) {
      const int it = e / (D / 4);
      const int k4 = e - it * (D / 4);
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (i0 + it < p.rows)
        v = *reinterpret_cast<const float4*>(p.table + static_cast<size_t>(i0 + it) * D + k4 * 4);
      reinterpret_cast<float4*>(sE)[e] = v;
    }
    if (tid < IT) sBias[tid] = p.bias_pad[i0 + tid];
    __syncthreads();

    for (int it = 0; it < IT; ++it) {
      const float4* e4 = reinterpret_cast<const float4*>(sE + it * D);
      // strict left-to-right fp32 accumulation in 4 interleaved partial sums keeps the result
      // within ~1e-7 relative of any other fp32 summation order.
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
      for (int k4 = 0; k4 < D / 4; ++k4) {
        const float4 ev = e4[k4];
        a0 = fmaf(u[4 * k4 + 0], ev.x, a0);
        a1 = fmaf(u[4 * k4 + 1], ev.y, a1);
        a2 = fmaf(u[4 * k4 + 2], ev.z, a2);
        a3 = fmaf(u[4 * k4 + 3], ev.w, a3);
      }
      const float s = ((a0 + a1) + (a2 + a3)) + sBias[it];
      if (kDense) {
        sOut[tid * (IT + 1) + it] = s;
      } else if (live && s >= own_thr) {
        const int gid = p.row_offset + i0 + it;
        const int bw = (gid >> 5) & 3;
        const uint32_t bword = bw == 0 ? bloom0 : (bw == 1 ? bloom1 : (bw == 2 ? bloom2 : bloom3));
        own_thr = tc::topk_consider<ROWS, LRB_MAX_K>(s, gid, limit_gid, own_thr, ls_a, li_a, ln_a, p.K, excl,
                                          p.excl_stride, bword);
      }
    }
    if (kDense) {
      __syncthreads();
      // coalesced write-out: 64 consecutive floats per row
      for (int e = tid; e < ROWS * IT; e += ROWS) {
        const int rr = e / IT;
        const int it = e - rr * IT;
        const int row = blockIdx.x * ROWS + rr;
        if (row < p.B && i0 + it < p.rows)
          p.dense_out[static_cast<size_t>(row) * p.dense_ld + i0 + it] = sOut[rr * (IT + 1) + it];
      }
    }
  }

  if (!kDense && live) {
    const int cnt = sCnt[tid];
    const size_t base = static_cast<size_t>(b) * p.slots + blockIdx.y;
    p.part_cnt[base] = cnt;
    for (int i = 0; i < cnt; ++i) {
      p.part_scores[base * p.K + i] = sListS[i * ROWS + tid];
      p.part_ids[base * p.K + i] = sListI[i * ROWS + tid];
    }
  }
}

inline int splits_for(int B, long long rows, int sms, int ctas_per_sm = 2) {
  const int m_tiles = (B + ROWS - 1) / ROWS;
  const long long chunks = (rows + IT - 1) / IT;
  long long want = (static_cast<long long>(ctas_per_sm) * sms + m_tiles - 1) / m_tiles;
  long long max_splits = (chunks + 3) / 4;   // at least 4 chunks (256 items) per split
  if (max_splits < 1) max_splits = 1;
  if (want > max_splits) want = max_splits;
  if (want < 1) want = 1;
  if (want > 1024) want = 1024;
  return static_cast<int>(want);
}

// --------------------------------------------------------------------------------------------
// Small catalogues: dense scores + per-user selection.
//
// The streaming kernel above keeps one top-K set per thread and pays a lock-step insertion for almost
// every item while a thread has seen fewer than ~32 K items (B200, C3 = 2048 users x 11001 items, K = 50:
// 875 us, of which the contraction itself is < 10 %, and 494 us more to merge 19 x 50 candidates per user).
// When a block of users' score rows fits in the scratch buffer the scores are written out once instead
// (score_f32_kernel<true>, same fp32 summation order) and ONE WARP PER USER selects the top K from its row:
//   1. the history mask as the reference applies it -- scores[b, history] = -inf (trainer/lru.py:36-38),
//   2. a 4-pass radix select (8 bits per pass, per-warp shared-memory histogram) for the K-th largest key,
//   3. one more pass collecting everything above the K-th key plus the lowest-id entries equal to it,
//   4. a rank sort of the <= K survivors into (score desc, id asc) order.
// The output is ONE sorted list per user (slots == 1), in the part_* layout the merge kernel consumes.
//
// Lists longer than 64 entries (K in [51, LRB_MAX_K_WIDE], CAP = 1024) take the wide variant of the kernel: the radix
// select runs on a 64-bit key (score key, then ~id), so the K selected entries are exactly the K best by
// (score desc, id asc) whatever order they are read in; it stops after the 8-bit pass whose bin holds exactly the
// entries still needed (the 4 score passes unless the K-th score is tied).  A warp-wide bitonic sort of the <= 1024
// survivors in shared memory replaces the rank sort.  Its loader is either a dense score row (implicit ids, as
// above) or an explicit candidate list of (score, id) pairs (kCand: the collect pass of the wide bf16 top-K,
// lrb_wide_select), whose history / out-of-shard ids are dropped first.
// --------------------------------------------------------------------------------------------
constexpr int SEL_WARPS = 8;
constexpr int SEL_WARPS_WIDE = 4;   // 4 x (4 KB histogram + 8 KB of 64-bit keys) = 48 KB of static shared memory
constexpr int SEL_CAP_WIDE = 1024;

struct SelParams {
  float* dense;          // [nb][ld] scores of this user block (scratch; the history mask is written into it)
  long long ld;
  int nb;                // users in the block
  int b0;                // global index of the block's first user
  int rows, row_offset, K;
  const int* excl_sorted;
  int excl_stride;
  float* part_scores;    // [B][K]
  int* part_ids;
  int* part_cnt;         // [B]
};

// the wide variant's parameters (K > 64), kept out of SelParams so that the K <= 64 kernel compiles as before
struct SelParamsWide : SelParams {
  const int* users;      // row i of the block belongs to user users[i] (null: user b0 + i)
  float* cand_scores;    // kCand: [nb][cap] collected (score, id) pairs, compacted in place
  int* cand_ids;
  const int* cand_cnt;   // [nb] collected items, also past cap
  int cap;
  int8_t* path;          // [B] (null: not written) ok_path / -1 overflow, tau_out valid / -2 short
  int ok_path;
  float* tau_out;        // [B] overflow: the K-th best admissible score among the stored pairs
};

LRB_DEVINL unsigned sel_key(float v) {   // order-preserving unsigned key; NaN sorts below everything
  return (v == v) ? (static_cast<unsigned>(float_to_key(v)) ^ 0x80000000u) : 0u;
}

template <int CAP, bool kCand, class Prm = SelParamsWide>
__global__ void __launch_bounds__((CAP <= 64 ? SEL_WARPS : SEL_WARPS_WIDE) * 32) select_topk_kernel(const Prm p);

// K <= 64 (CAP == 64): dense rows only
template <>
__global__ void __launch_bounds__(SEL_WARPS * 32) select_topk_kernel<64, false, SelParams>(const SelParams p) {
  __shared__ unsigned s_hist[SEL_WARPS][4 * 256];
  __shared__ float s_sc[SEL_WARPS][64];
  __shared__ int s_id[SEL_WARPS][64];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int bl = blockIdx.x * SEL_WARPS + warp;
  if (bl >= p.nb) return;                       // (no block-level barrier below)
  const int b = p.b0 + bl;
  float* row = p.dense + static_cast<size_t>(bl) * p.ld;
  const int rows = p.rows;
  unsigned* hist = s_hist[warp];
  const unsigned lt_mask = (1u << lane) - 1u;

  // 1. history mask
  if (p.excl_sorted != nullptr) {
    const int* ex = p.excl_sorted + static_cast<size_t>(b) * p.excl_stride;
    for (int j = lane; j < p.excl_stride; j += 32) {
      const int id = ex[j];
      const long long col = static_cast<long long>(id) - p.row_offset;
      if (id != INT_MAX && col >= 0 && col < rows) row[col] = -INFINITY;
    }
  }
  __syncwarp();

  // 2. radix select: the `need`-th largest key among the row's entries
  const int K_eff = p.K < rows ? p.K : rows;
  unsigned prefix = 0u;
  int need = K_eff;
#pragma unroll 1
  for (int pass = 0; pass < 4; ++pass) {
    const int shift = 24 - 8 * pass;
    const unsigned hi_mask = pass == 0 ? 0u : (0xffffffffu << (shift + 8));
#pragma unroll
    for (int j = 0; j < 32; ++j) hist[lane + 32 * j] = 0u;
    __syncwarp();
    // Four row entries per lane and iteration are loaded before any is counted (the loop is latency-bound: one
    // warp per user, ~14 resident warps per SM at C3), and the histogram exists in four copies selected by lane % 4:
    // scores share their sign and exponent bits, so in the first passes nearly every lane hits the same bin and
    // the shared-memory atomics serialise.  (Grouping the lanes with match.any instead was twice as slow.)
    unsigned* my_hist = hist + (lane & 3) * 256;
    for (int base = lane; base < rows; base += 128) {
      float v[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) v[q] = (base + 32 * q < rows) ? row[base + 32 * q] : 0.f;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const unsigned key = sel_key(v[q]);
        if (base + 32 * q < rows && (key & hi_mask) == prefix) atomicAdd(&my_hist[(key >> shift) & 255u], 1u);
      }
    }
    __syncwarp();
    // lane l owns bins [8l, 8l+8); `above` = entries in bins owned by higher lanes
    unsigned own[8];
    unsigned mine = 0u;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int bi = lane * 8 + j;
      own[j] = hist[bi] + hist[256 + bi] + hist[512 + bi] + hist[768 + bi];
      mine += own[j];
    }
    unsigned incl = mine;                       // inclusive suffix sum over lanes (high lanes first)
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned v = __shfl_down_sync(0xffffffffu, incl, o);
      if (lane + o < 32) incl += v;
    }
    const unsigned above = incl - mine;
    const bool holder = above < static_cast<unsigned>(need) && static_cast<unsigned>(need) <= incl;
    int bin = 0;
    unsigned above_bin = 0u;
    if (holder) {
      unsigned acc = above;
#pragma unroll
      for (int j = 7; j >= 0; --j) {
        if (acc < static_cast<unsigned>(need) && static_cast<unsigned>(need) <= acc + own[j]) { bin = lane * 8 + j; above_bin = acc; }
        acc += own[j];
      }
    }
    const unsigned hb = __ballot_sync(0xffffffffu, holder);
    const int src = __ffs(hb) - 1;              // exactly one holder (need >= 1 and need <= matching entries)
    bin = __shfl_sync(0xffffffffu, bin, src);
    above_bin = __shfl_sync(0xffffffffu, above_bin, src);
    prefix |= static_cast<unsigned>(bin) << shift;
    need -= static_cast<int>(above_bin);
    __syncwarp();
  }
  // prefix = key of the K-th largest entry; `need` entries equal to it are wanted (lowest columns first)
  const int n_gt_total = K_eff - need;

  // 3. collect (ballot prefix sums keep the equal-key entries in column order)
  int n_gt = 0, n_eq = 0;
  for (int base = 0; base < rows; base += 128) {
    float vv[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) vv[q] = (base + 32 * q + lane < rows) ? row[base + 32 * q + lane] : 0.f;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int c = base + 32 * q + lane;
      const bool valid = c < rows;
      const float v = vv[q];
      const unsigned key = valid ? sel_key(v) : 0u;
      const bool gt = valid && key > prefix;
      const bool eq = valid && key == prefix;
      const unsigned bg = __ballot_sync(0xffffffffu, gt);
      const unsigned be = __ballot_sync(0xffffffffu, eq);
      if (gt) {
        const int idx = n_gt + __popc(bg & lt_mask);
        s_sc[warp][idx] = v;
        s_id[warp][idx] = c + p.row_offset;
      }
      if (eq) {
        const int r = n_eq + __popc(be & lt_mask);
        if (r < need) {
          s_sc[warp][n_gt_total + r] = v;
          s_id[warp][n_gt_total + r] = c + p.row_offset;
        }
      }
      n_gt += __popc(bg);
      n_eq += __popc(be);
    }
    if (n_gt >= n_gt_total && n_eq >= need) break;   // warp-uniform
  }
  __syncwarp();

  // 4. rank sort into (score desc, id asc); -inf (masked / padding) and NaN entries are not emitted
  int n_valid = 0;
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const int e = lane + 32 * q;
    bool ok = false;
    int rank = 0;
    float sc = 0.f;
    int id = 0;
    if (e < K_eff) {
      sc = s_sc[warp][e];
      id = s_id[warp][e];
      ok = sc > -INFINITY;
      for (int j = 0; j < K_eff; ++j) {
        const float sj = s_sc[warp][j];
        const int ij = s_id[warp][j];
        rank += (sj > -INFINITY && better(sj, ij, sc, id)) ? 1 : 0;
      }
    }
    if (ok) {
      p.part_scores[static_cast<size_t>(b) * p.K + rank] = sc;
      p.part_ids[static_cast<size_t>(b) * p.K + rank] = id;
    }
    n_valid += __popc(__ballot_sync(0xffffffffu, ok));
  }
  if (lane == 0) p.part_cnt[b] = n_valid;
}

LRB_DEVINL unsigned long long sel_key64(float v, int id) {
  return (static_cast<unsigned long long>(sel_key(v)) << 32) | static_cast<unsigned>(~id);
}
LRB_DEVINL float sel_key_score(unsigned long long k) {
  return key_to_float(static_cast<int>(static_cast<unsigned>(k >> 32) ^ 0x80000000u));
}

template <int CAP, bool kCand, class Prm>
__global__ void __launch_bounds__(SEL_WARPS_WIDE * 32) select_topk_kernel(const Prm p) {
  static_assert(CAP == SEL_CAP_WIDE, "wide variant");
  __shared__ unsigned s_hist[SEL_WARPS_WIDE][4 * 256];
  __shared__ unsigned long long s_key[SEL_WARPS_WIDE][CAP];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int bl = blockIdx.x * SEL_WARPS_WIDE + warp;
  if (bl >= p.nb) return;                       // (no block-level barrier below)
  const int b = p.users != nullptr ? p.users[bl] : p.b0 + bl;
  const int* ex = p.excl_sorted != nullptr ? p.excl_sorted + static_cast<size_t>(b) * p.excl_stride : nullptr;
  unsigned* hist = s_hist[warp];
  unsigned long long* keys = s_key[warp];
  const unsigned lt_mask = (1u << lane) - 1u;

  // 1. loader: n entries, entry j = (score, id)
  float* row = nullptr;
  int* cid = nullptr;
  int n = 0, cnt = 0;
  if constexpr (kCand) {
    cnt = p.cand_cnt[bl];
    const int stored = cnt < p.cap ? cnt : p.cap;
    row = p.cand_scores + static_cast<size_t>(bl) * p.cap;
    cid = p.cand_ids + static_cast<size_t>(bl) * p.cap;
    // drop history ids and ids outside the shard (compaction in place: writes only to positions <= those read)
    for (int base = 0; base < stored; base += 32) {
      const int j = base + lane;
      const int id = j < stored ? cid[j] : -1;
      const float v = j < stored ? row[j] : 0.f;
      const long long local = static_cast<long long>(id) - p.row_offset;
      bool ok = j < stored && local >= 0 && local < p.rows;
      if (ok && ex != nullptr) {
        int lo = 0, hi = p.excl_stride;
        while (lo < hi) {
          const int mid = (lo + hi) >> 1;
          if (__ldg(ex + mid) < id) lo = mid + 1; else hi = mid;
        }
        ok = !(lo < p.excl_stride && __ldg(ex + lo) == id);
      }
      const unsigned bal = __ballot_sync(0xffffffffu, ok);
      __syncwarp();
      if (ok) {
        const int idx = n + __popc(bal & lt_mask);
        cid[idx] = id;
        row[idx] = v;
      }
      n += __popc(bal);
    }
  } else {
    row = p.dense + static_cast<size_t>(bl) * p.ld;
    n = p.rows;
    if (ex != nullptr) {                        // the history mask, as in the K <= 64 variant
      for (int j = lane; j < p.excl_stride; j += 32) {
        const int id = ex[j];
        const long long col = static_cast<long long>(id) - p.row_offset;
        if (id != INT_MAX && col >= 0 && col < n) row[col] = -INFINITY;
      }
    }
  }
  __syncwarp();
  auto key_at = [&](int j) -> unsigned long long {
    if constexpr (kCand) return sel_key64(row[j], cid[j]);
    else return sel_key64(row[j], j + p.row_offset);
  };

  // 2. radix select of the K_eff-th largest 64-bit key, 8 bits per pass
  const int K_eff = p.K < n ? p.K : n;
  unsigned long long prefix = 0ull;
  int need = K_eff;
  int bits = 0;                                 // leading key bits that decide: entries with top bits >= prefix's
#pragma unroll 1
  for (int pass = 0; pass < 8 && need > 0; ++pass) {
    const int shift = 56 - 8 * pass;
    const unsigned long long hi_mask = pass == 0 ? 0ull : (~0ull << (shift + 8));
#pragma unroll
    for (int j = 0; j < 32; ++j) hist[lane + 32 * j] = 0u;
    __syncwarp();
    unsigned* my_hist = hist + (lane & 3) * 256;
    for (int base = lane; base < n; base += 128) {
      unsigned long long kk[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) kk[q] = (base + 32 * q < n) ? key_at(base + 32 * q) : 0ull;
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (base + 32 * q < n && (kk[q] & hi_mask) == prefix)
          atomicAdd(&my_hist[static_cast<unsigned>(kk[q] >> shift) & 255u], 1u);
    }
    __syncwarp();
    unsigned own[8];
    unsigned mine = 0u;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int bi = lane * 8 + j;
      own[j] = hist[bi] + hist[256 + bi] + hist[512 + bi] + hist[768 + bi];
      mine += own[j];
    }
    unsigned incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned v = __shfl_down_sync(0xffffffffu, incl, o);
      if (lane + o < 32) incl += v;
    }
    const unsigned above = incl - mine;
    const bool holder = above < static_cast<unsigned>(need) && static_cast<unsigned>(need) <= incl;
    int bin = 0;
    unsigned above_bin = 0u, bin_cnt = 0u;
    if (holder) {
      unsigned acc = above;
#pragma unroll
      for (int j = 7; j >= 0; --j) {
        if (acc < static_cast<unsigned>(need) && static_cast<unsigned>(need) <= acc + own[j]) {
          bin = lane * 8 + j; above_bin = acc; bin_cnt = own[j];
        }
        acc += own[j];
      }
    }
    const int src = __ffs(__ballot_sync(0xffffffffu, holder)) - 1;
    bin = __shfl_sync(0xffffffffu, bin, src);
    above_bin = __shfl_sync(0xffffffffu, above_bin, src);
    bin_cnt = __shfl_sync(0xffffffffu, bin_cnt, src);
    prefix |= static_cast<unsigned long long>(bin) << shift;
    need -= static_cast<int>(above_bin);
    bits = 8 * (pass + 1);
    __syncwarp();
    if (bin_cnt == static_cast<unsigned>(need)) break;   // every entry of the bin is wanted (keys are distinct)
  }

  // 3. collect the K_eff entries whose leading `bits` bits reach the prefix's
  int ns = 0;
  if (K_eff > 0) {
    const int sh = 64 - bits;
    const unsigned long long thr = prefix >> sh;
    for (int base = 0; base < n; base += 128) {
      unsigned long long kk[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) kk[q] = (base + 32 * q + lane < n) ? key_at(base + 32 * q + lane) : 0ull;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const bool sel = base + 32 * q + lane < n && (kk[q] >> sh) >= thr;
        const unsigned bs = __ballot_sync(0xffffffffu, sel);
        const int idx = ns + __popc(bs & lt_mask);
        if (sel && idx < CAP) keys[idx] = kk[q];
        ns += __popc(bs);
      }
      if (ns >= K_eff) break;                   // warp-uniform
    }
    ns = ns < K_eff ? ns : K_eff;
  }
  // 4. bitonic sort (descending) of the survivors, padded with key 0 to a power of two
  int P = 32;
  while (P < ns) P <<= 1;
  for (int j = ns + lane; j < P; j += 32) keys[j] = 0ull;
  __syncwarp();
  for (int k = 2; k <= P; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = lane; i < P; i += 32) {
        const int ixj = i ^ j;
        if (ixj > i) {
          const unsigned long long a = keys[i], c = keys[ixj];
          if (((i & k) == 0) ? (a < c) : (a > c)) { keys[i] = c; keys[ixj] = a; }
        }
      }
      __syncwarp();
    }
  }
  // 5. -inf (masked / padding) and NaN entries sort last and are not emitted
  const unsigned long long lowest = static_cast<unsigned long long>(sel_key(-INFINITY)) << 32 | 0xffffffffull;
  int n_valid = 0;
  for (int base = 0; base < ns; base += 32) {
    const int j = base + lane;
    n_valid += __popc(__ballot_sync(0xffffffffu, j < ns && keys[j] > lowest));
  }
  int8_t st = static_cast<int8_t>(p.ok_path);
  if constexpr (kCand) {
    if (n_valid < p.K) st = -2;                 // short: tau was above the K-th best, or too few admissible items
    else if (cnt > p.cap) st = -1;              // overflow: retry at the K-th best stored score
  }
  if (st >= 0) {
    for (int j = lane; j < n_valid; j += 32) {
      const unsigned long long k = keys[j];
      p.part_scores[static_cast<size_t>(b) * p.K + j] = sel_key_score(k);
      p.part_ids[static_cast<size_t>(b) * p.K + j] = static_cast<int>(~static_cast<unsigned>(k));
    }
    if (lane == 0) p.part_cnt[b] = n_valid;
  }
  if (lane == 0) {
    if (p.path != nullptr) p.path[b] = st;
    if (st == -1) p.tau_out[b] = sel_key_score(keys[p.K - 1]);
  }
}

// users whose score rows fit in `bytes` of scratch (multiple of 128, the dense kernel's user tile), 0 = none
inline long long select_block_users(long long rows, size_t bytes) {
  const long long ld = (rows + 3) / 4 * 4;
  const long long u = static_cast<long long>(bytes / (static_cast<size_t>(ld) * 4));
  return u / ROWS * ROWS;
}

// dense fp32 scores out[M][ld] (columns < rows) of the user states x [M][64] against table [rows][64] + bias_pad
int launch_dense(const float* x, const float* table, const float* bias_pad, int M, int rows, float* out,
                 long long ld, int sms, cudaStream_t st) {
  Params p;
  p.u = x;
  p.table = table;
  p.bias_pad = bias_pad;
  p.B = M; p.rows = rows; p.row_offset = 0; p.K = 0;
  p.excl_sorted = nullptr; p.excl_bloom = nullptr; p.excl_stride = 0;
  p.part_scores = nullptr; p.part_ids = nullptr; p.part_cnt = nullptr; p.slots = 0;
  p.dense_out = out; p.dense_ld = ld;
  const int splits = splits_for(M, rows, sms, 4);   // dense variant: 49 KB / 96 registers -> 4 CTAs per SM
  const size_t smem = (IT * D + IT) * 4 + static_cast<size_t>(ROWS) * (IT + 1) * 4;
  auto kern = score_f32_kernel<true>;
  LRB_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  dim3 grid(static_cast<unsigned>((static_cast<long long>(M) + ROWS - 1) / ROWS), splits);
  kern<<<grid, ROWS, smem, st>>>(p);
  LRB_CUDA_TRY(cudaGetLastError());
  return LRB_OK;
}

}  // namespace f32

// ============================================================================================
// Wide top-K helpers (lrb_wide_sample_threshold)
// ============================================================================================
namespace wide {

__global__ void fill_kernel(float* out, int n, float v) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = v;
}

// The exclusion list of the lattice view (row i of the view = shard row r * i): shard-local ids divisible by r, as
// view rows, ascending and INT_MAX padded, with their bloom filter (the layout of lrb_prepare_sequences).  One warp
// per user.
__global__ void __launch_bounds__(256) lattice_excl_kernel(const int* excl, int stride, int B, int row_offset, int rows,
                                                           int r, int* out, uint32_t* bloom) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * 8 + warp;
  if (b >= B) return;
  const int* ex = excl + static_cast<size_t>(b) * stride;
  int* o = out + static_cast<size_t>(b) * stride;
  uint32_t w0 = 0u, w1 = 0u, w2 = 0u, w3 = 0u;
  int n = 0;
  for (int base = 0; base < stride; base += 32) {
    const int j = base + lane;
    const int id = j < stride ? ex[j] : INT_MAX;
    const long long local = static_cast<long long>(id) - row_offset;
    const bool ok = id != INT_MAX && local >= 0 && local < rows && local % r == 0;
    const int v = ok ? static_cast<int>(local / r) : 0;
    const unsigned bal = __ballot_sync(0xffffffffu, ok);
    if (ok) {
      o[n + __popc(bal & ((1u << lane) - 1u))] = v;
      const uint32_t bit = 1u << (v & 31);
      const int wd = (v >> 5) & 3;
      w0 |= wd == 0 ? bit : 0u; w1 |= wd == 1 ? bit : 0u; w2 |= wd == 2 ? bit : 0u; w3 |= wd == 3 ? bit : 0u;
    }
    n += __popc(bal);
  }
  for (int j = n + lane; j < stride; j += 32) o[j] = INT_MAX;
  w0 = __reduce_or_sync(0xffffffffu, w0); w1 = __reduce_or_sync(0xffffffffu, w1);
  w2 = __reduce_or_sync(0xffffffffu, w2); w3 = __reduce_or_sync(0xffffffffu, w3);
  if (lane == 0) reinterpret_cast<uint4*>(bloom)[b] = make_uint4(w0, w1, w2, w3);
}

}  // namespace wide

// ============================================================================================
// tcgen05 path: decomposition + tensor maps + launch
// ============================================================================================
namespace {

struct Decomp {
  int m_tiles, n_tiles, s_full, rem, full_tiles, y_tiles, grid, slots;
};

// `units` = independent MMA engines (SMs, or SM pairs when two CTAs share one tcgen05.mma), `bm` = users
// per engine tile (128 per CTA).
Decomp decompose(int B, long long rows, int units, int bm = tc::BM) {
  const int sms = units;
  Decomp d;
  d.m_tiles = (B + bm - 1) / bm;
  d.n_tiles = static_cast<int>((rows + tc::BN - 1) / tc::BN);
  long long work = static_cast<long long>(d.m_tiles) * d.n_tiles;
  int G = static_cast<int>(work < sms ? work : sms);
  if (G < 1) G = 1;
  d.s_full = G / d.m_tiles;
  d.rem = G - d.s_full * d.m_tiles;
  if (d.s_full == 0) {
    d.rem = G;
    d.y_tiles = d.n_tiles;
    d.full_tiles = 0;
  } else if (d.rem == 0) {
    d.y_tiles = 0;
    d.full_tiles = d.n_tiles;
  } else {
    // per-CTA work in item tiles: full stream = full_tiles / s_full ; shared stream = m_tiles * y / rem -- plus what
    // every (re)start of a streaming top-K costs (thresholds are weak at first: candidate appends and drains; measured
    // ~0.45M cycles for a full-stream segment; shared-stream segments start under the full streams' union bound and
    // are cheaper -- A/B on one B200: R0 = 0 / 150 / 300 / 600 tiles give 4.97 / 4.84 / 4.93 / 4.91 ms at 4096 x 10M
    // and 5.44 / 5.40 / 5.52 / 5.58 ms at 32768 x 1.25M, hence R0 = 150).  A full-stream CTA starts once, a
    // shared-stream CTA about m_tiles / rem + 1/2 times:
    //   (n - y) / s + R0  =  m * y / rem + (m / rem + 1/2) * R0
    double R0 = RESTART_TILES;
    if (R0 > d.n_tiles / (8.0 * d.s_full)) R0 = d.n_tiles / (8.0 * d.s_full);   // short segments: a start costs less
    const double m_over_rem = static_cast<double>(d.m_tiles) / d.rem;
    double y = (static_cast<double>(d.n_tiles) / d.s_full + R0 * (0.5 - m_over_rem)) / (1.0 / d.s_full + m_over_rem);
    if (y < 0.0) y = 0.0;
    d.y_tiles = static_cast<int>(std::floor(y + 0.5));
    if (d.y_tiles > d.n_tiles) d.y_tiles = d.n_tiles;
    if (d.y_tiles <= 0) { d.y_tiles = 0; d.rem = 0; }
    d.full_tiles = d.n_tiles - d.y_tiles;
  }
  d.grid = d.s_full * d.m_tiles + d.rem;
  d.slots = tc::PARTS * (d.s_full + (d.rem > 0 ? 2 : 0));
  return d;
}

// Users per launch.  A streaming top-K restarts for every (launch, item range) and its start-up is the
// expensive part (thresholds are weak until a few thousand items have been seen), so large batches -- the
// all-gathered users of a data-parallel job -- want few, long segments; but the union bound needs
// c * 2 * s_full >= K with c <= MAX_C_SHARE entries per stream, and a launch whose user tiles divide the SM
// pairs evenly has no remainder ("shared") stream.  148 SMs: 37 pair tiles = 9472 users per launch, two full
// streams per user, c = 5.  Measured on B200 (debug build, 32768 users x 1.25M rows): launches of 4096 users
// 8.85 ms, 5632: 8.70, 8192: 8.39, 9472 (+ one of 4352): 8.30, 18944 (no union bound): 10.2.
inline int users_per_launch(int B, int sms) {
  const int units = sms >= 2 ? sms / 2 : 1;                 // CTA pairs
  // one pair tile (256 users) per CTA pair: every user has ONE full stream over the whole local item range, so each
  // streaming top-K restarts once (two slots per user, union bound with c = ceil(K/2) <= 12).  Measured on B200,
  // 32768 users x 1.25M rows (one rank's call of the 8-GPU data-parallel step): launches of 9472 users (two full
  // streams, c = 5) 5.58 ms, of 18944 users 5.38 ms.
  const int cap = units * 2 * tc::BM;
  return B <= cap ? B : cap;
}

// CTA pairs (tcgen05 cta_group::2) whenever a launch has more than one user tile: the pair shares every
// item tile, which halves the shared-memory operand traffic and the L2 -> SM traffic per MMA.
inline int cta_group_for(int B, int sms) { return (B > tc::BM && sms >= 2) ? 2 : 1; }

Decomp decompose_launch(int B, long long rows, int sms) {
  const int cg = cta_group_for(B, sms);
  return decompose(B, rows, sms / cg, tc::BM * cg);
}

int chunked_slots(int B, long long rows, int sms) {
  const int cap = users_per_launch(B, sms);
  int slots = 0;
  for (int c0 = 0; c0 < B; c0 += cap) {
    const int s = decompose_launch(B - c0 < cap ? B - c0 : cap, rows, sms).slots;
    slots = s > slots ? s : slots;
  }
  return slots;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
    tried = true;
  }
  return fn;
}

// [rows][64] bf16 row-major, box = 64 x box_rows, 128-byte swizzle, OOB rows read as zero.  row_bytes > 128: a
// strided view (every (row_bytes / 128)-th row of the table, the lattice sample of the wide top-K).
int make_tmap_bf16_k64(CUtensorMap* out, const void* ptr, unsigned long long rows, unsigned box_rows,
                       unsigned long long row_bytes = 128ull) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return set_error(LRB_ERR_DRIVER, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[2] = {64ull, rows};
  cuuint64_t strides[1] = {row_bytes};
  cuuint32_t box[2] = {64u, box_rows};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides,
                  box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error(LRB_ERR_DRIVER, "cuTensorMapEncodeTiled failed (%d)", (int)r);
  return LRB_OK;
}

// folded-bias block: row-major [n_tiles * 256][16] bf16 (32 B per item), box = 16 x box_rows (the whole tile, or a CTA
// pair's 128-row half), 32-byte swizzle.  row_bytes > 32: the strided view over `view_rows` items that goes with a
// strided table view (rows past view_rows read as zero; the kernels mask those columns by their index).
int make_tmap_bias_blocks(CUtensorMap* out, const void* ptr, unsigned long long n_tiles, unsigned box_rows,
                          unsigned long long row_bytes = 32ull, unsigned long long view_rows = 0ull) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return set_error(LRB_ERR_DRIVER, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[2] = {16ull, row_bytes == 32ull ? n_tiles * tc::BN : view_rows};
  cuuint64_t strides[1] = {row_bytes};
  cuuint32_t box[2] = {16u, box_rows};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error(LRB_ERR_DRIVER, "cuTensorMapEncodeTiled (bias blocks) failed (%d)", (int)r);
  return LRB_OK;
}

// `grid` counts MMA engines: CTAs for CG == 1, CTA pairs (clusters of 2) for CG == 2.
template <int KMAX, int NS, bool kDense, int CG, int CMAX = tc::MAX_C_SHARE_SMALL, bool kCollect = false,
          bool kCollectScores = false>
int launch_tc(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tbias, const tc::ScoreParams& p,
              int grid, cudaStream_t st, bool overlap_prev = false) {
  using L = tc::SmemLayout<KMAX, NS, CG>;
  auto kern = tc::score_topk_tc_kernel<KMAX, NS, kDense, CG, CMAX, kCollect, kCollectScores>;
  LRB_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::kAlloc));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(static_cast<unsigned>(grid * CG));
  cfg.blockDim = dim3(128 + tc::EPI_WARPS * 32);
  cfg.dynamicSmemBytes = L::kAlloc;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (CG > 1) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = CG;
    attr[na].val.clusterDim.y = 1;
    attr[na].val.clusterDim.z = 1;
    ++na;
  }
  if (overlap_prev) {   // may start while the previous chunk launch is still draining (see the kernel prologue)
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  cfg.attrs = attr;
  cfg.numAttrs = na;
  LRB_CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, ta, tb, tbias, p));
  LRB_CUDA_TRY(cudaGetLastError());
  return LRB_OK;
}

}  // namespace
}  // namespace lrb

extern "C" {

static size_t ring_bytes();
// users per block of the exact-fp32 "dense + select" path (0 = the catalogue is too large for it): what fits in
// the candidate-ring part of the scratch buffer, which lrb_score_scratch_bytes() reserves for every B
static long long f32_select_users(long long rows) { return lrb::f32::select_block_users(rows, 2 * ring_bytes()); }
// the largest shard the dense + select path takes (one 128-user block of score rows in the scratch)
static long long f32_select_rows_max() {
  return static_cast<long long>(2 * ring_bytes() / (lrb::f32::ROWS * sizeof(float))) / 4 * 4;
}

int lrb_score_topk_slots(int B, int64_t rows, int precision, int* slots) {
  LRB_REQUIRE(B > 0 && rows > 0 && slots != nullptr, "lrb_score_topk_slots: bad arguments");
  int sms = lrb::device_sm_count();
  if (sms <= 0) sms = 148;
  if (precision == 0) {
    *slots = lrb::chunked_slots(B, rows, sms);
  } else if (precision == 1) {
    // small catalogues: dense scores + per-user selection -> one sorted list per user
    *slots = f32_select_users(rows) > 0 ? 1 : lrb::f32::splits_for(B, rows, sms);
  } else {
    return lrb::set_error(LRB_ERR_BAD_ARG, "precision must be 0 (bf16) or 1 (fp32)");
  }
  return LRB_OK;
}

// worst-case slot count is 2 * (number of SMs + 2): reserve that so the size depends on B only
static size_t gslots_bytes(int B) {
  int sms = lrb::device_sm_count();
  if (sms <= 0) sms = 148;
  size_t m_tiles = (static_cast<size_t>(B) + lrb::tc::BM - 1) / lrb::tc::BM;
  if (m_tiles > static_cast<size_t>(sms)) m_tiles = static_cast<size_t>(sms);   // one launch never covers more
  const size_t max_slots = lrb::tc::PARTS * (static_cast<size_t>(sms) / m_tiles + 2);
  // (+1 tile: CTA pairs pad the user tiles to an even count)
  return ((m_tiles + 1) * lrb::tc::BM * max_slots * sizeof(int) + 255) & ~static_cast<size_t>(255);
}

// union-bound slots of one chunk launch of at most `cap` users (the worst case over smaller chunks: few user
// tiles mean many streams, i.e. many slots per user)
static size_t gslots_chunk_bytes(int cap) {
  size_t mx = 0;
  for (int b = lrb::tc::BM; b < cap + lrb::tc::BM; b += lrb::tc::BM) {
    const size_t v = gslots_bytes(b < cap ? b : cap);
    mx = v > mx ? v : mx;
  }
  return mx;
}

static size_t ring_bytes() {
  int sms = lrb::device_sm_count();
  if (sms <= 0) sms = 148;
  // 512 rings per SM, twice the kernel's 256 epilogue threads; the size also sets the user block of the fp32 select
  // path (f32_select_users), so it is part of the dispatch
  return static_cast<size_t>(sms) * 512 * lrb::tc::RING_GROUPS * lrb::tc::RING_REC_BYTES;
}

// layout: [n_chunks x union-bound slots of one chunk][2 x candidate rings (consecutive chunk launches overlap)]
size_t lrb_score_scratch_bytes(int B) {
  int sms = lrb::device_sm_count();
  if (sms <= 0) sms = 148;
  if (B < 1) B = 1;
  const int cap = lrb::users_per_launch(B, sms);
  const size_t n_chunks = (static_cast<size_t>(B) + cap - 1) / cap;
  return n_chunks * gslots_chunk_bytes(cap) + 2 * ring_bytes();
}

// The bf16 streaming top-K of lrb_score_topk over `rows` item rows; r > 1: over the strided view of every r-th row of
// table / bias_blk (local row i = table row r * i), the lattice sample of lrb_wide_sample_threshold.
static int topk_bf16(const void* u, const void* table, const void* bias_blk, int B, int64_t rows, int64_t row_offset,
                     const int32_t* excl_sorted, const uint32_t* excl_bloom, int excl_stride, int K,
                     float* part_scores, int32_t* part_ids, int32_t* part_cnt, int slots, void* scratch,
                     cudaStream_t st, int sms, int r) {
  using namespace lrb;
  CUtensorMap tb1, tb2, tbias, tbias1;
  const unsigned long long tstride = 128ull * r, bstride = 32ull * r;
  int rc = make_tmap_bf16_k64(&tb1, table, static_cast<unsigned long long>(rows), tc::BN, tstride);
  if (rc != LRB_OK) return rc;
  rc = make_tmap_bf16_k64(&tb2, table, static_cast<unsigned long long>(rows), tc::BN / 2, tstride);
  if (rc != LRB_OK) return rc;
  tbias = tb1;   // placeholders when there is no bias block (never dereferenced)
  tbias1 = tb1;
  if (bias_blk != nullptr) {
    const unsigned long long nt = static_cast<unsigned long long>((rows + tc::BN - 1) / tc::BN);
    rc = make_tmap_bias_blocks(&tbias, bias_blk, nt, tc::BN / 2, bstride, rows);     // a CTA pair's halves
    if (rc != LRB_OK) return rc;
    rc = make_tmap_bias_blocks(&tbias1, bias_blk, nt, tc::BN, bstride, rows);        // single CTAs: the whole tile
    if (rc != LRB_OK) return rc;
  }
  LRB_CUDA_TRY(cudaMemsetAsync(part_cnt, 0, static_cast<size_t>(B) * slots * sizeof(int), st));
  const int cap = users_per_launch(B, sms);
  const size_t n_chunks = (static_cast<size_t>(B) + cap - 1) / cap;
  const size_t gs_chunk = gslots_chunk_bytes(cap);
  // every chunk's union-bound slots are reset up front: nothing but kernels between the chunk launches
  LRB_CUDA_TRY(cudaMemsetAsync(scratch, 0x80, n_chunks * gs_chunk, st));
  int chunk_idx = 0;
  int prev_ctas = 0;
  for (int c0 = 0; c0 < B; c0 += cap, ++chunk_idx) {
    // one launch per user chunk (see users_per_launch); chunk-relative pointers
    const int Bc = B - c0 < cap ? B - c0 : cap;
    const int cg = cta_group_for(Bc, sms);
    const Decomp d = decompose_launch(Bc, rows, sms);
    CUtensorMap ta;
    rc = make_tmap_bf16_k64(&ta, static_cast<const uint8_t*>(u) + static_cast<size_t>(c0) * 128,
                            static_cast<unsigned long long>(Bc), tc::BM);
    if (rc != LRB_OK) return rc;
    tc::ScoreParams p;
    p.B = Bc; p.m_tiles = d.m_tiles; p.rows = static_cast<int>(rows); p.n_tiles = d.n_tiles;
    p.row_offset = static_cast<int>(row_offset); p.K = K;
    p.bias_blk = static_cast<const uint8_t*>(bias_blk);
    p.excl_sorted = excl_sorted ? excl_sorted + static_cast<size_t>(c0) * excl_stride : nullptr;
    p.excl_bloom = excl_bloom ? excl_bloom + static_cast<size_t>(c0) * 4 : nullptr;
    p.excl_stride = excl_stride;
    p.gslots = reinterpret_cast<int*>(static_cast<uint8_t*>(scratch) + chunk_idx * gs_chunk);
    p.gstride = d.slots;
    p.ring = static_cast<uint8_t*>(scratch) + n_chunks * gs_chunk + (chunk_idx & 1) * ring_bytes();
    {
      // entries each of the PARTS*s_full full-stream threads of a user must hold for the union bound
      const int c = d.s_full > 0 ? (K + tc::PARTS * d.s_full - 1) / (tc::PARTS * d.s_full) : 99;
      // (the K <= 20 CTA-pair kernel also exists with room for c <= 12: one full stream per user)
      const int c_max = (cg == 2 && K <= 20) ? tc::MAX_C_SHARE_LARGE : tc::MAX_C_SHARE_SMALL;
      p.c_share = c <= c_max ? c : 0;
      // scout pass: worth its T0 extra tiles when the union bound exists and segments are long enough
      const long long seg_tiles = d.s_full > 0 ? d.full_tiles / d.s_full : 0;
      // (32 tiles on long segments: A/B on B200, 32768 users x 1.25M rows -- one stream per user, c = 10 --
      // 16 / 32 / 64 scout tiles give 4.95 / 4.79 / 4.90 ms; 4096 x 10M is indifferent within run-to-run noise)
      p.scout_tiles = (p.c_share > 0 && seg_tiles >= 128) ? (seg_tiles >= 512 ? 32 : 16) : 0;
    }
    p.part_scores = part_scores + static_cast<size_t>(c0) * slots * K;
    p.part_ids = part_ids + static_cast<size_t>(c0) * slots * K;
    p.part_cnt = part_cnt + static_cast<size_t>(c0) * slots;
    p.slots = slots;
    p.dense_out = nullptr; p.dense_ld = 0;
    p.s_full = d.s_full; p.rem = d.rem; p.full_tiles = d.full_tiles; p.y_tiles = d.y_tiles;
    // Overlap with the previous chunk launch is safe for the scratch as long as chunk i never runs next to
    // chunk i-2 (they share a ring copy): one CTA fits per SM, so that cannot happen when chunk i-1 fills
    // every SM -- chunk i can then only start once chunk i-2 is gone.
    const bool ov = chunk_idx == 1 || (chunk_idx > 1 && prev_ctas >= sms);
    prev_ctas = d.grid * cg;
    if (cg == 2) {
      if (K <= 20 && p.c_share > tc::MAX_C_SHARE_SMALL)
        rc = launch_tc<20, NS_PAIR, false, 2, tc::MAX_C_SHARE_LARGE>(ta, tb2, tbias, p, d.grid, st, ov);
      else if (K <= 20) rc = launch_tc<20, NS_PAIR, false, 2>(ta, tb2, tbias, p, d.grid, st, ov);
      else if (K <= 32) rc = launch_tc<32, 4, false, 2>(ta, tb2, tbias, p, d.grid, st, ov);
      else rc = launch_tc<50, 3, false, 2>(ta, tb2, tbias, p, d.grid, st, ov);
    } else {
      if (K <= 20) rc = launch_tc<20, 2, false, 1>(ta, tb1, tbias1, p, d.grid, st, ov);
      else if (K <= 32) rc = launch_tc<32, 3, false, 1>(ta, tb1, tbias1, p, d.grid, st, ov);
      else rc = launch_tc<50, 2, false, 1>(ta, tb1, tbias1, p, d.grid, st, ov);
    }
    if (rc != LRB_OK) return rc;
  }
  return LRB_OK;
}

int lrb_score_topk(const void* u, const void* table, const float* bias_pad, const void* bias_blk,
                   int B, int64_t rows,
                   int64_t row_offset, const int32_t* excl_sorted, const uint32_t* excl_bloom,
                   int excl_stride, int K, int precision, float* part_scores, int32_t* part_ids,
                   int32_t* part_cnt, int slots, void* scratch, void* stream) {
  using namespace lrb;
  int rc = check_arch();
  if (rc != LRB_OK) return rc;
  LRB_REQUIRE(u && table && part_scores && part_ids && part_cnt, "lrb_score_topk: null pointer");
  LRB_REQUIRE(precision != 1 || bias_pad != nullptr, "lrb_score_topk: the fp32 path needs bias_pad");
  LRB_REQUIRE(B > 0 && rows > 0 && rows + row_offset < INT_MAX, "lrb_score_topk: bad B/rows");
  LRB_REQUIRE(K >= 1 && K <= LRB_MAX_K_WIDE, "lrb_score_topk: K must be in [1, %d]", LRB_MAX_K_WIDE);
  LRB_REQUIRE(K <= LRB_MAX_K || K <= rows, "lrb_score_topk: K=%d > %d needs K <= rows (%lld)", K, LRB_MAX_K,
              static_cast<long long>(rows));
  LRB_REQUIRE((excl_sorted == nullptr) == (excl_bloom == nullptr), "lrb_score_topk: exclusion list and bloom filter must come together");
  if (K > LRB_MAX_K && !(precision == 1 && f32_select_users(rows) > 0))
    return set_error(LRB_ERR_UNSUPPORTED, "lrb_score_topk: K=%d > %d only on the fp32 dense + select path "
                     "(rows <= %lld); use lrb_wide_* for bf16", K, LRB_MAX_K, f32_select_rows_max());
  cudaStream_t st = as_stream(stream);
  int sms = device_sm_count();
  if (precision == 1 && f32_select_users(rows) > 0) {
    LRB_REQUIRE(slots == 1, "lrb_score_topk: slots=%d but lrb_score_topk_slots says 1", slots);
    LRB_REQUIRE(scratch != nullptr, "lrb_score_topk: scratch is required");
    const long long blk = f32_select_users(rows);
    const long long ld = (rows + 3) / 4 * 4;
    float* dense = static_cast<float*>(scratch);
    for (long long b0 = 0; b0 < B; b0 += blk) {
      const int nb = static_cast<int>(B - b0 < blk ? B - b0 : blk);
      rc = f32::launch_dense(static_cast<const float*>(u) + b0 * f32::D, static_cast<const float*>(table), bias_pad,
                             nb, static_cast<int>(rows), dense, ld, sms, st);
      if (rc != LRB_OK) return rc;
      f32::SelParams sp;
      sp.dense = dense; sp.ld = ld; sp.nb = nb; sp.b0 = static_cast<int>(b0);
      sp.rows = static_cast<int>(rows); sp.row_offset = static_cast<int>(row_offset); sp.K = K;
      sp.excl_sorted = excl_sorted; sp.excl_stride = excl_stride;
      sp.part_scores = part_scores; sp.part_ids = part_ids; sp.part_cnt = part_cnt;
      if (K <= LRB_MAX_K) {
        f32::select_topk_kernel<64, false, f32::SelParams><<<(nb + f32::SEL_WARPS - 1) / f32::SEL_WARPS, f32::SEL_WARPS * 32, 0, st>>>(sp);
      } else {
        f32::SelParamsWide wp = {};
        static_cast<f32::SelParams&>(wp) = sp;
        f32::select_topk_kernel<f32::SEL_CAP_WIDE, false>
            <<<(nb + f32::SEL_WARPS_WIDE - 1) / f32::SEL_WARPS_WIDE, f32::SEL_WARPS_WIDE * 32, 0, st>>>(wp);
      }
      LRB_CUDA_TRY(cudaGetLastError());
    }
    return LRB_OK;
  }
  if (precision == 1) {
    const int splits = f32::splits_for(B, rows, sms);
    LRB_REQUIRE(slots == splits, "lrb_score_topk: slots=%d but lrb_score_topk_slots says %d", slots, splits);
    f32::Params p;
    p.u = static_cast<const float*>(u);
    p.table = static_cast<const float*>(table);
    p.bias_pad = bias_pad;
    p.B = B; p.rows = static_cast<int>(rows); p.row_offset = static_cast<int>(row_offset); p.K = K;
    p.excl_sorted = excl_sorted; p.excl_bloom = excl_bloom; p.excl_stride = excl_stride;
    p.part_scores = part_scores; p.part_ids = part_ids; p.part_cnt = part_cnt; p.slots = slots;
    p.dense_out = nullptr; p.dense_ld = 0;
    const size_t smem = (f32::IT * f32::D + f32::IT) * 4 + static_cast<size_t>(K) * f32::ROWS * 8;
    auto kern = f32::score_f32_kernel<false>;
    LRB_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    dim3 grid((B + f32::ROWS - 1) / f32::ROWS, splits);
    kern<<<grid, f32::ROWS, smem, st>>>(p);
    LRB_CUDA_TRY(cudaGetLastError());
    return LRB_OK;
  }
  LRB_REQUIRE(precision == 0, "precision must be 0 (bf16) or 1 (fp32)");
  LRB_REQUIRE(scratch != nullptr, "lrb_score_topk: scratch is required for the bf16 path");
  const int want_slots = chunked_slots(B, rows, sms);
  LRB_REQUIRE(slots == want_slots, "lrb_score_topk: slots=%d but lrb_score_topk_slots says %d", slots, want_slots);
  return topk_bf16(u, table, bias_blk, B, rows, row_offset, excl_sorted, excl_bloom, excl_stride, K, part_scores,
                   part_ids, part_cnt, slots, scratch, st, sms, 1);
}

int lrb_score_dense(const void* x, const void* table, const float* bias_pad, const void* bias_blk,
                    int64_t M, int64_t rows, int precision, float* out, int64_t ld_out, void* stream) {
  using namespace lrb;
  int rc = check_arch();
  if (rc != LRB_OK) return rc;
  LRB_REQUIRE(x && table && out, "lrb_score_dense: null pointer");
  LRB_REQUIRE(precision != 1 || bias_pad != nullptr, "lrb_score_dense: the fp32 path needs bias_pad");
  LRB_REQUIRE(M > 0 && M < INT_MAX && rows > 0 && rows < INT_MAX && ld_out >= rows, "lrb_score_dense: bad shape");
  cudaStream_t st = as_stream(stream);
  int sms = device_sm_count();
  if (precision == 1)
    return f32::launch_dense(static_cast<const float*>(x), static_cast<const float*>(table), bias_pad,
                             static_cast<int>(M), static_cast<int>(rows), out, ld_out, sms, st);
  LRB_REQUIRE(precision == 0, "precision must be 0 (bf16) or 1 (fp32)");
  const Decomp d = decompose(static_cast<int>(M), rows, sms);
  CUtensorMap ta, tb;
  rc = make_tmap_bf16_k64(&ta, x, static_cast<unsigned long long>(M), tc::BM);
  if (rc != LRB_OK) return rc;
  rc = make_tmap_bf16_k64(&tb, table, static_cast<unsigned long long>(rows), tc::BN);
  if (rc != LRB_OK) return rc;
  tc::ScoreParams p;
  p.B = static_cast<int>(M); p.m_tiles = d.m_tiles; p.rows = static_cast<int>(rows); p.n_tiles = d.n_tiles;
  p.row_offset = 0; p.K = 1; p.bias_blk = static_cast<const uint8_t*>(bias_blk);
  p.excl_sorted = nullptr; p.excl_bloom = nullptr; p.excl_stride = 0;
  p.gslots = nullptr; p.gstride = 0; p.c_share = 0; p.scout_tiles = 0; p.ring = nullptr; p.part_scores = nullptr; p.part_ids = nullptr; p.part_cnt = nullptr; p.slots = 0;
  p.dense_out = out; p.dense_ld = ld_out;
  p.s_full = d.s_full; p.rem = d.rem; p.full_tiles = d.full_tiles; p.y_tiles = d.y_tiles;
  CUtensorMap tbias = tb;   // placeholder without a bias block (never dereferenced)
  if (bias_blk != nullptr) {
    rc = make_tmap_bias_blocks(&tbias, bias_blk, static_cast<unsigned long long>((rows + tc::BN - 1) / tc::BN), tc::BN);
    if (rc != LRB_OK) return rc;
  }
  return launch_tc<20, 3, true, 1>(ta, tb, tbias, p, d.grid, st);
}

static int collect_impl(const void* u_bf16, const void* table_bf16, const void* bias_blk, int M, int64_t rows,
                        int64_t row_offset, const float* tau, int cap, int32_t* cand_ids, float* cand_scores,
                        int32_t* cand_cnt, void* stream) {
  using namespace lrb;
  int rc = check_arch();
  if (rc != LRB_OK) return rc;
  LRB_REQUIRE(u_bf16 && table_bf16 && tau && cand_cnt, "lrb_score_collect: null pointer");
  LRB_REQUIRE(cap >= 0 && (cap == 0 || cand_ids != nullptr), "lrb_score_collect: bad cap / cand_ids");
  LRB_REQUIRE(M > 0 && rows > 0 && rows + row_offset < INT_MAX && row_offset >= 0, "lrb_score_collect: bad shape");
  cudaStream_t st = as_stream(stream);
  const int sms = device_sm_count();
  // the dense mode's decomposition and launch shape (one CTA per tile, no CTA pairs): the collect pass differs
  // from it only in the epilogue
  const Decomp d = decompose(M, rows, sms);
  CUtensorMap ta, tb;
  rc = make_tmap_bf16_k64(&ta, u_bf16, static_cast<unsigned long long>(M), tc::BM);
  if (rc != LRB_OK) return rc;
  rc = make_tmap_bf16_k64(&tb, table_bf16, static_cast<unsigned long long>(rows), tc::BN);
  if (rc != LRB_OK) return rc;
  CUtensorMap tbias = tb;   // placeholder without a bias block (never dereferenced)
  if (bias_blk != nullptr) {
    rc = make_tmap_bias_blocks(&tbias, bias_blk, static_cast<unsigned long long>((rows + tc::BN - 1) / tc::BN), tc::BN);
    if (rc != LRB_OK) return rc;
  }
  tc::ScoreParams p = {};
  p.B = M; p.m_tiles = d.m_tiles; p.rows = static_cast<int>(rows); p.n_tiles = d.n_tiles;
  p.row_offset = static_cast<int>(row_offset); p.K = 1; p.bias_blk = static_cast<const uint8_t*>(bias_blk);
  p.s_full = d.s_full; p.rem = d.rem; p.full_tiles = d.full_tiles; p.y_tiles = d.y_tiles;
  p.collect_tau = tau; p.collect_ids = cand_ids; p.collect_cnt = cand_cnt; p.collect_cap = cap;
  p.collect_scores = cand_scores;
  LRB_CUDA_TRY(cudaMemsetAsync(cand_cnt, 0, static_cast<size_t>(M) * sizeof(int32_t), st));
  if (cand_scores != nullptr)
    return launch_tc<20, 3, true, 1, tc::MAX_C_SHARE_SMALL, true, true>(ta, tb, tbias, p, d.grid, st);
  return launch_tc<20, 3, true, 1, tc::MAX_C_SHARE_SMALL, true>(ta, tb, tbias, p, d.grid, st);
}

int lrb_score_collect(const void* u_bf16, const void* table_bf16, const void* bias_blk, int M, int64_t rows,
                      int64_t row_offset, const float* tau, int cap, int32_t* cand_ids, int32_t* cand_cnt,
                      void* stream) {
  return collect_impl(u_bf16, table_bf16, bias_blk, M, rows, row_offset, tau, cap, cand_ids, nullptr, cand_cnt,
                      stream);
}

int lrb_score_collect_scores(const void* u_bf16, const void* table_bf16, const void* bias_blk, int M, int64_t rows,
                             int64_t row_offset, const float* tau, int cap, int32_t* cand_ids, float* cand_scores,
                             int32_t* cand_cnt, void* stream) {
  LRB_REQUIRE(cap == 0 || cand_scores != nullptr, "lrb_score_collect_scores: null cand_scores");
  return collect_impl(u_bf16, table_bf16, bias_blk, M, rows, row_offset, tau, cap, cand_ids, cand_scores, cand_cnt,
                      stream);
}

// ---- wide top-K (K in [51, LRB_MAX_K_WIDE]) on the bf16 path ----------------------------------------------------

static size_t align256(size_t x) { return (x + 255) & ~static_cast<size_t>(255); }

struct SampleLayout {
  long long n_lat;
  int slots;
  size_t excl, bloom, part_s, part_i, part_c, top_s, top_i, scratch, total;
};

static SampleLayout sample_layout(int B, int64_t rows, int excl_stride, int r, int m) {
  SampleLayout L = {};
  int sms = lrb::device_sm_count();
  if (sms <= 0) sms = 148;
  L.n_lat = (rows + r - 1) / r;
  L.slots = lrb::chunked_slots(B, L.n_lat, sms);
  const size_t Bs = static_cast<size_t>(B);
  size_t o = 0;
  L.excl = o;    o += align256(Bs * (excl_stride > 0 ? excl_stride : 0) * 4);
  L.bloom = o;   o += align256(Bs * 16);
  L.part_s = o;  o += align256(Bs * L.slots * m * 4);
  L.part_i = o;  o += align256(Bs * L.slots * m * 4);
  L.part_c = o;  o += align256(Bs * L.slots * 4);
  L.top_s = o;   o += align256(Bs * m * 4);
  L.top_i = o;   o += align256(Bs * m * 4);
  L.scratch = o; o += align256(lrb_score_scratch_bytes(B));
  L.total = o;
  return L;
}

size_t lrb_wide_sample_workspace_bytes(int B, int64_t rows, int excl_stride, int r, int m) {
  if (B < 1 || rows < 1 || r < 1 || m < 1 || m > LRB_MAX_K) return 256;
  return sample_layout(B, rows, excl_stride, r, m).total;
}

int lrb_wide_sample_threshold(const void* u_bf16, const void* table_bf16, const void* bias_blk, int B, int64_t rows,
                              int64_t row_offset, const int32_t* excl_sorted, int excl_stride, int r, int m,
                              float* tau, void* workspace, size_t workspace_bytes, void* stream) {
  using namespace lrb;
  int rc = check_arch();
  if (rc != LRB_OK) return rc;
  LRB_REQUIRE(u_bf16 && table_bf16 && tau && workspace, "lrb_wide_sample_threshold: null pointer");
  LRB_REQUIRE(B > 0 && rows > 0 && row_offset >= 0 && rows + row_offset < INT_MAX,
              "lrb_wide_sample_threshold: bad shape");
  LRB_REQUIRE(r >= 1 && r <= (1 << 20) && m >= 1 && m <= LRB_MAX_K,
              "lrb_wide_sample_threshold: need r in [1, 2^20] and m in [1, %d]", LRB_MAX_K);
  LRB_REQUIRE(excl_sorted == nullptr || excl_stride > 0, "lrb_wide_sample_threshold: bad excl_stride");
  const SampleLayout L = sample_layout(B, rows, excl_sorted ? excl_stride : 0, r, m);
  if (workspace_bytes < L.total)
    return set_error(LRB_ERR_WORKSPACE, "lrb_wide_sample_threshold: workspace %zu < %zu bytes", workspace_bytes,
                     L.total);
  cudaStream_t st = as_stream(stream);
  if (L.n_lat < m) {                            // fewer than m lattice rows: no threshold
    wide::fill_kernel<<<(B + 255) / 256, 256, 0, st>>>(tau, B, -INFINITY);
    LRB_CUDA_TRY(cudaGetLastError());
    return LRB_OK;
  }
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  int32_t* excl = nullptr;
  uint32_t* bloom = nullptr;
  if (excl_sorted != nullptr) {
    excl = reinterpret_cast<int32_t*>(ws + L.excl);
    bloom = reinterpret_cast<uint32_t*>(ws + L.bloom);
    wide::lattice_excl_kernel<<<(B + 7) / 8, 256, 0, st>>>(excl_sorted, excl_stride, B, static_cast<int>(row_offset),
                                                           static_cast<int>(rows), r, excl, bloom);
    LRB_CUDA_TRY(cudaGetLastError());
  }
  float* part_s = reinterpret_cast<float*>(ws + L.part_s);
  int32_t* part_i = reinterpret_cast<int32_t*>(ws + L.part_i);
  int32_t* part_c = reinterpret_cast<int32_t*>(ws + L.part_c);
  rc = topk_bf16(u_bf16, table_bf16, bias_blk, B, L.n_lat, 0, excl, bloom, excl_stride, m, part_s, part_i, part_c,
                 L.slots, ws + L.scratch, st, device_sm_count(), r);
  if (rc != LRB_OK) return rc;
  float* top_s = reinterpret_cast<float*>(ws + L.top_s);
  rc = lrb_merge_metrics(part_s, part_i, part_c, L.slots, m, static_cast<int64_t>(L.slots) * m, 1, L.slots, m, B, m,
                         nullptr, nullptr, 0, top_s, reinterpret_cast<int32_t*>(ws + L.top_i), 0, nullptr, nullptr,
                         stream);
  if (rc != LRB_OK) return rc;
  // tau = the m-th entry of the merged lattice list (-inf when the lattice holds fewer than m admissible rows)
  LRB_CUDA_TRY(cudaMemcpy2DAsync(tau, sizeof(float), top_s + (m - 1), static_cast<size_t>(m) * sizeof(float),
                                 sizeof(float), static_cast<size_t>(B), cudaMemcpyDeviceToDevice, st));
  return LRB_OK;
}

// dense bf16 rows of the wide select's fallback: users per block so that a block of rows stays near 1 GiB
static long long wide_dense_block(int64_t rows) {
  const long long ld = (rows + 3) / 4 * 4;
  const long long blk = (1ll << 30) / (ld * 4);
  return blk < 1 ? 1 : blk;
}

size_t lrb_wide_select_workspace_bytes(int n, int64_t rows) {
  if (n < 1 || rows < 1) return 256;
  const long long ld = (rows + 3) / 4 * 4;
  const long long blk = wide_dense_block(rows);
  return align256(static_cast<size_t>(n < blk ? n : blk) * ld * sizeof(float));
}

int lrb_wide_select(const int32_t* users, int n, const void* u_bf16, const void* table_bf16, const void* bias_blk,
                    int64_t rows, int64_t row_offset, const int32_t* excl_sorted, int excl_stride, float* cand_scores,
                    int32_t* cand_ids, const int32_t* cand_cnt, int cap, int K, int ok_path, float* out_scores,
                    int32_t* out_ids, int32_t* out_cnt, int8_t* path, float* tau_out, void* workspace,
                    size_t workspace_bytes, void* stream) {
  using namespace lrb;
  int rc = check_arch();
  if (rc != LRB_OK) return rc;
  LRB_REQUIRE(users && out_scores && out_ids && out_cnt && path, "lrb_wide_select: null pointer");
  LRB_REQUIRE(n > 0 && rows > 0 && row_offset >= 0 && rows + row_offset < INT_MAX, "lrb_wide_select: bad shape");
  LRB_REQUIRE(K >= 1 && K <= LRB_MAX_K_WIDE, "lrb_wide_select: K must be in [1, %d]", LRB_MAX_K_WIDE);
  LRB_REQUIRE(K <= rows, "lrb_wide_select: K=%d > rows (%lld)", K, static_cast<long long>(rows));
  LRB_REQUIRE(ok_path >= 0 && ok_path <= 127, "lrb_wide_select: ok_path must be in [0, 127]");
  LRB_REQUIRE(excl_sorted == nullptr || excl_stride > 0, "lrb_wide_select: bad excl_stride");
  cudaStream_t st = as_stream(stream);
  f32::SelParamsWide sp = {};
  sp.rows = static_cast<int>(rows); sp.row_offset = static_cast<int>(row_offset); sp.K = K;
  sp.excl_sorted = excl_sorted; sp.excl_stride = excl_stride;
  sp.part_scores = out_scores; sp.part_ids = out_ids; sp.part_cnt = out_cnt;
  sp.path = path; sp.ok_path = ok_path; sp.tau_out = tau_out;
  constexpr int W = f32::SEL_WARPS_WIDE;
  if (cand_scores != nullptr) {                 // explicit candidate lists
    LRB_REQUIRE(cand_ids && cand_cnt && tau_out && cap >= 1, "lrb_wide_select: candidate lists need ids, counts, "
                "tau_out and cap >= 1");
    sp.nb = n; sp.users = users;
    sp.cand_scores = cand_scores; sp.cand_ids = cand_ids; sp.cand_cnt = cand_cnt; sp.cap = cap;
    f32::select_topk_kernel<f32::SEL_CAP_WIDE, true><<<(n + W - 1) / W, W * 32, 0, st>>>(sp);
    LRB_CUDA_TRY(cudaGetLastError());
    return LRB_OK;
  }
  // dense bf16 rows (lrb_score_dense precision 0) of u_bf16 row i = user users[i], in blocks of the workspace
  LRB_REQUIRE(u_bf16 && table_bf16 && workspace, "lrb_wide_select: the dense loader needs u_bf16, table and workspace");
  const size_t need = lrb_wide_select_workspace_bytes(n, rows);
  if (workspace_bytes < need)
    return set_error(LRB_ERR_WORKSPACE, "lrb_wide_select: workspace %zu < %zu bytes", workspace_bytes, need);
  const long long ld = (rows + 3) / 4 * 4;
  const long long blk = wide_dense_block(rows);
  float* dense = static_cast<float*>(workspace);
  for (long long i0 = 0; i0 < n; i0 += blk) {
    const int nb = static_cast<int>(n - i0 < blk ? n - i0 : blk);
    rc = lrb_score_dense(static_cast<const uint8_t*>(u_bf16) + i0 * 128, table_bf16, nullptr, bias_blk, nb, rows, 0,
                         dense, ld, stream);
    if (rc != LRB_OK) return rc;
    sp.dense = dense; sp.ld = ld; sp.nb = nb; sp.users = users + i0;
    f32::select_topk_kernel<f32::SEL_CAP_WIDE, false><<<(nb + W - 1) / W, W * 32, 0, st>>>(sp);
    LRB_CUDA_TRY(cudaGetLastError());
  }
  return LRB_OK;
}

}  // extern "C"
