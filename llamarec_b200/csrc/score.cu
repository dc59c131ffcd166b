// Host launchers for catalogue scoring (+ the exact-fp32 FFMA variant for small catalogues).
//   lrb_score_topk   precision 0 -> score_topk_tc_kernel (tcgen05/TMEM/TMA, bf16 operands)
//                    precision 1 -> score_topk_f32_kernel (fp32 FFMA, bit-comparable with the
//                                   fp32 reference `x @ E^T + bias`, model/lru.py:85)
//   lrb_score_dense  API-compatible dense logits for LRURec.forward
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
// --------------------------------------------------------------------------------------------
constexpr int SEL_WARPS = 8;

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

LRB_DEVINL unsigned sel_key(float v) {   // order-preserving unsigned key; NaN sorts below everything
  return (v == v) ? (static_cast<unsigned>(float_to_key(v)) ^ 0x80000000u) : 0u;
}

__global__ void __launch_bounds__(SEL_WARPS * 32) select_topk_kernel(const SelParams p) {
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

// [rows][64] bf16 row-major, box = 64 x box_rows, 128-byte swizzle, OOB rows read as zero.
int make_tmap_bf16_k64(CUtensorMap* out, const void* ptr, unsigned long long rows, unsigned box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return set_error(LRB_ERR_DRIVER, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[2] = {64ull, rows};
  cuuint64_t strides[1] = {128ull};
  cuuint32_t box[2] = {64u, box_rows};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides,
                  box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error(LRB_ERR_DRIVER, "cuTensorMapEncodeTiled failed (%d)", (int)r);
  return LRB_OK;
}

// folded-bias block: row-major [n_tiles * 256][16] bf16 (32 B per item), box = 16 x box_rows (the whole tile, or a CTA
// pair's 128-row half), 32-byte swizzle
int make_tmap_bias_blocks(CUtensorMap* out, const void* ptr, unsigned long long n_tiles, unsigned box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return set_error(LRB_ERR_DRIVER, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[2] = {16ull, n_tiles * tc::BN};
  cuuint64_t strides[1] = {32ull};
  cuuint32_t box[2] = {16u, box_rows};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error(LRB_ERR_DRIVER, "cuTensorMapEncodeTiled (bias blocks) failed (%d)", (int)r);
  return LRB_OK;
}

// `grid` counts MMA engines: CTAs for CG == 1, CTA pairs (clusters of 2) for CG == 2.
template <int KMAX, int NS, bool kDense, int CG, int CMAX = tc::MAX_C_SHARE_SMALL>
int launch_tc(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tbias, const tc::ScoreParams& p,
              int grid, cudaStream_t st, bool overlap_prev = false) {
  using L = tc::SmemLayout<KMAX, NS, CG>;
  auto kern = tc::score_topk_tc_kernel<KMAX, NS, kDense, CG, CMAX>;
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
  LRB_REQUIRE(K >= 1 && K <= LRB_MAX_K, "lrb_score_topk: K must be in [1, %d]", LRB_MAX_K);
  LRB_REQUIRE((excl_sorted == nullptr) == (excl_bloom == nullptr), "lrb_score_topk: exclusion list and bloom filter must come together");
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
      f32::select_topk_kernel<<<(nb + f32::SEL_WARPS - 1) / f32::SEL_WARPS, f32::SEL_WARPS * 32, 0, st>>>(sp);
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
  CUtensorMap tb1, tb2, tbias, tbias1;
  rc = make_tmap_bf16_k64(&tb1, table, static_cast<unsigned long long>(rows), tc::BN);
  if (rc != LRB_OK) return rc;
  rc = make_tmap_bf16_k64(&tb2, table, static_cast<unsigned long long>(rows), tc::BN / 2);
  if (rc != LRB_OK) return rc;
  tbias = tb1;   // placeholders when there is no bias block (never dereferenced)
  tbias1 = tb1;
  if (bias_blk != nullptr) {
    const unsigned long long nt = static_cast<unsigned long long>((rows + tc::BN - 1) / tc::BN);
    rc = make_tmap_bias_blocks(&tbias, bias_blk, nt, tc::BN / 2);     // a CTA pair's halves
    if (rc != LRB_OK) return rc;
    rc = make_tmap_bias_blocks(&tbias1, bias_blk, nt, tc::BN);        // single CTAs: the whole tile
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

}  // extern "C"
