// Full-catalogue scoring fused with a streaming per-user top-K  (north_star subsystem 2).
//
// Replaces, for the last position only, the reference chain
//     scores = x @ E^T + bias                      model/lru.py:85
//     scores[b, history] = -1e9 ; scores[:,0]=-1e9 trainer/lru.py:36-38
//     torch.topk(scores, k)                        trainer/lru.py:82-84
// with one persistent sm_100a kernel:
//     TMA (SWIZZLE_128B)  ->  tcgen05.mma kind::f16 (bf16 x bf16 -> fp32 in TMEM)
//     ->  tcgen05.ld epilogue: group max (FMNMX3), threshold filter, rare slow path = dump the
//         16-score group to a ring; rings are drained warp-wide (lock-step) into per-thread top-K sets.
// The B x N score matrix never leaves the SM.
//
// Tile: 128 users (TMEM lanes) x 256 items x K=64 per CTA, staged in shared memory as one TMA tile and computed as
// two N = 128 half-tiles; FOUR TMEM accumulator stages of 128 columns.
// CG = 2 (every launch with more than one user tile): two CTAs of a TPC form a pair (cluster of 2,
// tcgen05 cta_group::2) that shares each 256-item tile -- every CTA stages only its 128 item rows, the leader
// issues M = 256 MMAs, both CTAs read their own 128-lane accumulators out of their own TMEM.
// Warp roles (384 threads): warp 0 = TMA producer, warps 1-2 = MMA issuers (leader CTA only; even / odd tiles),
// warp 2 also allocates TMEM, warp 3 = builds the "ones" block, then threshold service (union bound),
// warps 4..11 = epilogue (warp w reads TMEM lanes 32*(w%4).. of ONE half-tile per tile: warps 4-7 the first, warps
// 8-11 the second).  The
// producer / MMA / service warpgroup gives registers to the epilogue warpgroups (setmaxnreg 56 / 224).  The bias is
// folded into the GEMM as a fifth K=16 MMA per half-tile.  Consecutive launches of one call (user chunks) overlap via
// programmatic dependent launch.
#pragma once

#include <cuda.h>
#include "common.cuh"

namespace lrb {
namespace tc {

constexpr int BM = 128;
constexpr int BN = 256;
constexpr int BK = 64;
constexpr int A_BYTES = BM * BK * 2;
constexpr int B_BYTES = BN * BK * 2;
// The measurements quoted below that cite tools/tc_check, its probe builds ("MMA-only probe") or its
// timeline were taken with a developer harness that instrumented this kernel through extra template modes.  The
// harness has been removed; it is in the git history.
// Accumulators: the SM's 512 TMEM columns hold FOUR stages of 128 columns; a 256-item tile is computed as two
// N = 128 half-tiles.  With two 256-column stages the loop  release -> MMA -> commit -> read-out  ran ~1040 cycles per
// tile although the tensor pipe needs 512 and the read-out ~700: the hand-offs between the MMA-issuing thread and the
// epilogue warps (mbarrier round trips, remote arrivals of the pair's other CTA, MMA issue) add ~900 cycles to every
// stage cycle and only two stages were in flight to hide them (B200, tools/tc_check per-CTA counters: the epilogue
// warps AND the MMA warps waited for each other).  Four half-size stages double the work in flight.
constexpr int HN = 128;                     // accumulator columns per half-tile
constexpr int ACC_STAGES = 4;
constexpr int TMEM_COLS = ACC_STAGES * HN;
constexpr int DONE_RING = 8;                // tiles in the ring of "half-tile computed" barriers (two per tile); must exceed the TMA ring depth
// Epilogue warps: 8 (two column parts).  A 16-warp variant (four 64-column parts) was measured on B200 with the
// two-stage kernel of early round 2 (10M rows, 4096 users): it read the accumulators a little faster in isolation
// (tools/epi_probe: 702 vs 757 cycles per tile) but lost in the kernel (96 registers per thread, twice the per-thread
// candidate sets): 5.86 vs 5.25 ms; the kernel below is written for 8.
constexpr int EPI_WARPS = 8;
// Column parts of the epilogue = partial-list / union-bound slots per stream.  The two parts do not split every
// half-tile's columns (64 + 64) but take one half-tile each (part p reads all 128 columns of half-tile p): a stage is
// then released by 4 warps per CTA instead of 8, every warp waits / releases once per tile instead of twice, and the
// two warps of an SM sub-partition use its TMEM read path at different times.  Same-box A/B on B200 (tools/tc_check,
// product build): 4.76-4.91 -> 4.46-4.58 ms at 4096 x 10M, 5.07-5.31 -> 4.90-4.97 with bias + exclusion,
// 5.16-5.22 -> 4.95 at 32768 x 1.25M.
constexpr int PARTS = EPI_WARPS / 4;

struct ScoreParams {
  int B;             // real users (rows >= B of the padded user matrix are ignored)
  int m_tiles;       // padded users / 128
  int rows;          // real local item rows
  int n_tiles;       // ceil(rows / 256)
  int row_offset;    // global item id of local row 0
  int K;             // list length (<= KMAX)
  const uint8_t* bias_blk;     // folded bias: row-major [n_tiles * 256][16] bf16 (col 0..2 = hi/mid/lo split of the
                               // bias, -inf in col 0 beyond `rows`), fetched through tmap_bias with the 32-byte
                               // swizzle; nullptr = bias is identically zero
  const int* excl_sorted;      // [B][excl_stride] ascending global ids, INT_MAX padded; null = none
  const uint32_t* excl_bloom;  // [B][4] 128-bit membership filter over (id & 127)
  int excl_stride;
  int* gslots;                 // [m_tiles*128][slots] ordered-int keys: each FULL-stream thread's c-th best
                               // score so far (memset 0x80 = unset).  The PARTS*s_full full-stream slots of a
                               // user all start at t = 0; with c * PARTS*s_full >= K the minimum over them is a
                               // valid lower bound on the user's K-th best (union bound), also used by the
                               // shared-stream CTAs, whose own slots are ignored (they may start late).
  int c_share;                 // c (1..MAX_C_SHARE); 0 disables the union bound
  int scout_tiles;             // T0: the last T0 tiles of every segment are first run in "scout" mode (no
                               // candidate handling, only group maxima) to seed the union bound; 0 = off
  uint8_t* ring;               // [gridDim.x][epilogue threads][RING_GROUPS][RING_REC_BYTES] candidate rings
  float* part_scores;          // [B][slots][K]
  int* part_ids;               // [B][slots][K]
  int* part_cnt;               // [B][slots]   (zeroed by the host wrapper)
  int slots;                   // stride (in lists) of the part_* arrays
  int gstride;                 // stride (in ints) of gslots rows: the slot count of THIS launch
  float* dense_out;            // dense mode only: [B][dense_ld], columns < rows written
  long long dense_ld;
  // stream decomposition (host computed, see score_decompose())
  int s_full;        // number of full streams (each = m_tiles CTAs, one per user tile)
  int rem;           // CTAs in the shared stream
  int full_tiles;    // item tiles covered by the full streams  [0, full_tiles)
  int y_tiles;       // item tiles covered by the shared stream [full_tiles, n_tiles)
};

struct Segment {
  int m;      // user tile
  int n0;     // first item tile
  int n1;     // one past the last item tile
  int slot;   // stream slot (partial-list slot = slot * PARTS + column part)
};

// Deterministic walk over the segments owned by one CTA; every warp role runs the same walk.
struct SegmentWalk {
  int full;              // 1 = CTA belongs to a full stream
  int m, n0, n1, slot;   // the single segment of a full-stream CTA
  long long w, w_end;    // flattened (m * y + j) range of a shared-stream CTA
  int y, nbase, s_full;
  bool done;

  __device__ SegmentWalk(const ScoreParams& p, int cta) {
    s_full = p.s_full;
    y = p.y_tiles;
    nbase = p.full_tiles;
    done = false;
    if (cta < p.s_full * p.m_tiles) {
      full = 1;
      int s = cta / p.m_tiles;
      m = cta - s * p.m_tiles;
      n0 = static_cast<int>((static_cast<long long>(s) * p.full_tiles) / p.s_full);
      n1 = static_cast<int>((static_cast<long long>(s + 1) * p.full_tiles) / p.s_full);
      slot = s;
      w = w_end = 0;
    } else {
      full = 0;
      int j = cta - p.s_full * p.m_tiles;
      long long total = static_cast<long long>(p.m_tiles) * p.y_tiles;
      w = (total * j) / p.rem;
      w_end = (total * (j + 1)) / p.rem;
      m = n0 = n1 = slot = 0;
    }
  }
  __device__ bool next(Segment& s) {
    if (done) return false;
    if (full) {
      done = true;
      if (n1 <= n0) return false;
      s.m = m; s.n0 = n0; s.n1 = n1; s.slot = slot;
      return true;
    }
    if (w >= w_end) { done = true; return false; }
    int mm = static_cast<int>(w / y);
    int j0 = static_cast<int>(w - static_cast<long long>(mm) * y);
    long long len = y - j0;
    if (len > w_end - w) len = w_end - w;
    s.m = mm;
    s.n0 = nbase + j0;
    s.n1 = nbase + j0 + static_cast<int>(len);
    s.slot = s_full + (j0 != 0 ? 1 : 0);
    w += len;
    return true;
  }
};

// -------------------------------------------------------------------------------------------
// Slow path: one score that passed the threshold filter.  Checks bounds and the exclusion list,
// then offers it to this thread's candidate set: an UNSORTED array of K (score,id) pairs in shared
// memory (entry i at base + i*STRIDE*4) with the position of the worst entry cached, so that an
// accepted candidate costs one overwrite plus one rescan of K independent loads (no dependent
// shift chain).  ln[0] = entries held, ln[STRIDE] = index of the worst entry.
// Returns the thread's own K-th best score (-inf while the set is not full).
// All pointers are 32-bit shared-space addresses.
// -------------------------------------------------------------------------------------------
template <int STRIDE, int KMAX>
LRB_DEVINL float topk_consider_inl(float s, int gid, int row_limit_gid, float own_thr,
                                   uint32_t ls, uint32_t li, uint32_t ln, int K,
                                   const int* excl, uint32_t excl_s, int excl_stride,
                                   uint32_t bloom_word) {
  if (gid >= row_limit_gid) return own_thr;   // padded item column
  if (!(s == s)) return own_thr;              // NaN never ranks
  if (excl != nullptr && ((bloom_word >> (gid & 31)) & 1u)) {
    int lo = 0, hi = excl_stride;
    if (excl_s != 0u) {   // shared-memory copy of this row's sorted exclusion list
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (lds_s32(excl_s + mid * 4) < gid) lo = mid + 1; else hi = mid;
      }
      if (lo < excl_stride && lds_s32(excl_s + lo * 4) == gid) return own_thr;
    } else {
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(excl + mid) < gid) lo = mid + 1; else hi = mid;
      }
      if (lo < excl_stride && __ldg(excl + lo) == gid) return own_thr;  // in the user's history
    }
  }
  constexpr uint32_t ES = STRIDE * 4;  // byte stride between consecutive entries
  const int n = lds_s32(ln);
  if (n < K) {
    sts_f32(ls + n * ES, s);
    sts_s32(li + n * ES, gid);
    sts_s32(ln, n + 1);
    if (n + 1 < K) return -INFINITY;
  } else {
    const int wp = lds_s32(ln + ES);
    const float ws = lds_f32(ls + wp * ES);
    const int wi = lds_s32(li + wp * ES);
    if (!better(s, gid, ws, wi)) return own_thr;
    sts_f32(ls + wp * ES, s);
    sts_s32(li + wp * ES, gid);
  }
  // rescan: worst = lowest score, ties broken towards the higher id.  All K score loads are issued
  // back to back (independent), the minimum and its position are found without branches; ids are
  // only consulted when the minimum is not unique (rare).
  // (log-depth reductions: this runs in lock-step for the whole warp, its dependent-instruction depth is its cost)
  float v[KMAX];
#pragma unroll
  for (int i = 0; i < KMAX; ++i) v[i] = i < K ? lds_f32(ls + i * ES) : INFINITY;
  const float m = tree_min<KMAX>(v);
  int pos[KMAX], one[KMAX];
#pragma unroll
  for (int i = 0; i < KMAX; ++i) {
    const bool eq = v[i] == m;
    pos[i] = eq ? i : KMAX;
    one[i] = eq ? 1 : 0;
  }
  int mp = tree_min_int<KMAX>(pos);       // lowest position holding the minimum
  const int ties = tree_sum_int<KMAX>(one);
  if (mp >= KMAX) mp = 0;                 // (only if the minimum is a NaN, which never enters a set)
  if (ties > 1) {
    int mi = lds_s32(li + mp * ES);
    for (int i = mp + 1; i < K; ++i) {
      if (lds_f32(ls + i * ES) == m) {
        const int vi = lds_s32(li + i * ES);
        if (vi > mi) { mi = vi; mp = i; }
      }
    }
  }
  sts_s32(ln + ES, mp);
  return m;
}

template <int STRIDE, int KMAX>
__device__ __noinline__ float topk_consider(float s, int gid, int row_limit_gid, float own_thr,
                                            uint32_t ls, uint32_t li, uint32_t ln, int K,
                                            const int* excl, int excl_stride, uint32_t bloom_word) {
  return topk_consider_inl<STRIDE, KMAX>(s, gid, row_limit_gid, own_thr, ls, li, ln, K, excl, 0u, excl_stride,
                                   bloom_word);
}

// -------------------------------------------------------------------------------------------
// Deferred candidates.  When the maximum of a 16-score group reaches the thread's threshold the
// thread does NOT look at the individual scores: it dumps the group (16 floats + the global id of
// its first column) into a private ring in global memory (L2 resident, RING_GROUPS records of
// RING_REC_BYTES) and moves on -- 5 stores on a path that typically has a single active lane.
// The ring is drained by compact_ring(), which the whole warp enters together (lock-step): every
// lane repeatedly picks the best remaining score of its current record with a branch-free argmax
// and all lanes insert at the same time, so the insert cost is paid once per warp, not per lane.
// -------------------------------------------------------------------------------------------
constexpr int RING_GROUPS = 24;
constexpr int RING_REC_BYTES = 80;   // 16 fp32 + int32 gid0, padded to a multiple of 16 B

// c-th largest score of an unsorted set (1 <= c <= MAX_C_SHARE); -inf if the set holds fewer than c entries.
// MAX_C_SHARE (kernel template parameter CMAX) is 6 for launches whose users have >= 4 full-stream slots and 12 for
// the large launches of the data-parallel multi-GPU step (one full stream = 2 slots per user, c = 10 at K = 20).
constexpr int MAX_C_SHARE_SMALL = 6;
constexpr int MAX_C_SHARE_LARGE = 12;
template <int STRIDE, int MAX_C_SHARE>
LRB_DEVINL float set_cth_best(uint32_t ls, uint32_t ln, int c) {
  const int n = lds_s32(ln);
  float m[MAX_C_SHARE];   // running top-MAX_C_SHARE, descending
#pragma unroll
  for (int j = 0; j < MAX_C_SHARE; ++j) m[j] = -INFINITY;
  for (int i = 0; i < n; ++i) {
    float v = lds_f32(ls + i * STRIDE * 4);
#pragma unroll
    for (int j = 0; j < MAX_C_SHARE; ++j) {
      const float t = fminf(m[j], v);
      m[j] = fmaxf(m[j], v);
      v = t;
    }
  }
  float r = -INFINITY;
#pragma unroll
  for (int j = 0; j < MAX_C_SHARE; ++j) r = (c == j + 1) ? m[j] : r;
  return r;
}

struct RingRec {
  float4 a, b, c, d;
  int gid0;
};
LRB_DEVINL RingRec load_rec(const float4* ring, int g, bool act) {
  RingRec r;
  if (act) {
    const float4* rec = ring + g * (RING_REC_BYTES / 16);
    r.a = rec[0]; r.b = rec[1]; r.c = rec[2]; r.d = rec[3];
    r.gid0 = reinterpret_cast<const int*>(rec + 4)[0];
  } else {
    const float4 ninf = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    r.a = ninf; r.b = ninf; r.c = ninf; r.d = ninf;
    r.gid0 = 0;
  }
  return r;
}

template <int STRIDE, int KMAX>
__device__ __noinline__ float compact_ring(const float4* ring, int cnt, float own_thr, float shared_thr,
                                           int row_limit_gid, uint32_t ls, uint32_t li, uint32_t ln,
                                           int K, const int* excl, uint32_t excl_s, int excl_stride,
                                           uint32_t bloom0, uint32_t bloom1, uint32_t bloom2,
                                           uint32_t bloom3) {
  const int max_cnt = __reduce_max_sync(0xffffffffu, cnt);
  RingRec nxt = load_rec(ring, 0, 0 < cnt);
  for (int g = 0; g < max_cnt; ++g) {
    const bool act = g < cnt;
    const RingRec cur = nxt;
    nxt = load_rec(ring, g + 1, g + 1 < cnt);   // prefetch while this record is processed
    float s[16];
    const int gid0 = cur.gid0;
    s[0] = cur.a.x; s[1] = cur.a.y; s[2] = cur.a.z; s[3] = cur.a.w;
    s[4] = cur.b.x; s[5] = cur.b.y; s[6] = cur.b.z; s[7] = cur.b.w;
    s[8] = cur.c.x; s[9] = cur.c.y; s[10] = cur.c.z; s[11] = cur.c.w;
    s[12] = cur.d.x; s[13] = cur.d.y; s[14] = cur.d.z; s[15] = cur.d.w;
    while (true) {
      // best remaining score of the record and its lowest column (lower id wins ties); NaNs never win
      const float best = tree_max<16>(s);
      int col[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) col[j] = (s[j] == best) ? j : 16;
      const int bj = tree_min_int<16>(col) & 15;
      const bool pass = act && best > -INFINITY && best >= fmaxf(own_thr, shared_thr);
      if (!__any_sync(0xffffffffu, pass)) break;
      if (pass) {
        const int gid = gid0 + bj;
        const int bw = (gid >> 5) & 3;
        const uint32_t bword = bw == 0 ? bloom0 : (bw == 1 ? bloom1 : (bw == 2 ? bloom2 : bloom3));
        own_thr = topk_consider_inl<STRIDE, KMAX>(best, gid, row_limit_gid, own_thr, ls, li, ln, K, excl,
                                            excl_s, excl_stride, bword);
      }
#pragma unroll
      for (int j = 0; j < 16; ++j) s[j] = (pass && j == bj) ? -INFINITY : s[j];
    }
  }
  return own_thr;
}

// Everything only the drain needs, kept out of the hot loop's registers: the struct lives in the thread's local
// memory (its address is handed to the out-of-line drain_rings()), so that the filter loop holds little more than
// its two TMEM load buffers, the ring cursor and the threshold.
struct DrainState {
  const float4* ring;
  const int* excl;             // this row's sorted exclusion list in global memory (nullptr = none)
  int* rowthr;                 // this row's shared threshold (generic pointer into shared memory)
  int* gslot;                  // where this thread publishes its c-th best (nullptr = it does not)
  uint32_t excl_s;             // shared-memory copy of the list (0 = none)
  uint32_t bloom0, bloom1, bloom2, bloom3;
  uint32_t ls, li, ln;
  int excl_stride, K, limit_gid, c_share, published;
  bool live;
};

// Lock-step drain of the warp's rings (compact_ring) + publication of the improved bounds.  Returns the thread's
// own K-th best.
template <int STRIDE, int KMAX, int CMAX>
__device__ __noinline__ float drain_rings(DrainState* st, int cnt, float own_thr) {
  float shared_thr = -INFINITY;
  if (st->live) {
    const int kk = *reinterpret_cast<volatile int*>(st->rowthr);
    if (kk != INT_MIN) shared_thr = key_to_float(kk);
  }
  own_thr = compact_ring<STRIDE, KMAX>(st->ring, cnt, own_thr, shared_thr, st->limit_gid, st->ls, st->li, st->ln, st->K,
                                       st->excl, st->excl_s, st->excl_stride, st->bloom0, st->bloom1, st->bloom2,
                                       st->bloom3);
  if (st->live) {
    if (own_thr > -INFINITY) atomicMax(st->rowthr, float_to_key(own_thr));   // sibling column half
    if (st->gslot != nullptr) {
      const float cb = set_cth_best<STRIDE, CMAX>(st->ls, st->ln, st->c_share);
      const int key = float_to_key(cb);
      if (cb > -INFINITY && key > st->published) {
        st->published = key;
        *st->gslot = key;   // monotone, single writer
      }
    }
  }
  return own_thr;
}

constexpr int EX_CAP = 56;   // ints per row of the shared-memory exclusion copy (L <= 54)
constexpr int BIASBLK_BYTES = BN * 16 * 2;   // one tile of the folded-bias K=16 block (8 KB)
constexpr int ONES_BYTES = BM * 16 * 2;      // the matching [128][16] "ones" A block (4 KB)

// CG = CTAs per MMA (tcgen05 cta_group): with CG == 2 every CTA stages only its half of the item tile
// (128 rows) and of the bias block; the pair's MMA reads both halves.
// Epilogue warp w reads TMEM lanes 32*(w%4).. of half-tile (column part) w/4.
template <int KMAX, int NS, int CG>
struct SmemLayout {
  static constexpr int kEpiThreads = EPI_WARPS * 32;
  static constexpr bool kExclSmem = (KMAX <= 20);   // larger K variants have no room for it
  static constexpr int kBBytes = B_BYTES / CG;              // this CTA's part of the item tile
  static constexpr int kBiasBytes = BIASBLK_BYTES / CG;     // ... and of the folded-bias block
  static constexpr int kStage = kBBytes + kBiasBytes;
  static constexpr int kA = 0;
  static constexpr int kOnes = kA + A_BYTES;
  static constexpr int kB = kOnes + ONES_BYTES;            // 20 KB offset: 1024-aligned
  static constexpr int kListS = kB + NS * kStage;
  static constexpr int kListI = kListS + KMAX * kEpiThreads * 4;
  static constexpr int kListN = kListI + KMAX * kEpiThreads * 4;
  static constexpr int kRowThr = kListN + kEpiThreads * 8;
  static constexpr int kExcl = kRowThr + 2 * BM * 4 + 16;   // two threshold buffers + service-warp flags
  static constexpr int kBars = kExcl + (kExclSmem ? BM * EX_CAP * 4 : 0);
  // barriers: full[NS], done[DONE_RING][2], tmem_empty[ACC_STAGES], a_full, a_empty
  static constexpr int kNumBars = NS + 2 * DONE_RING + ACC_STAGES + 2;
  static constexpr int kTmemPtr = kBars + kNumBars * 8;
  static constexpr int kTotal = kTmemPtr + 16;
  static constexpr int kAlloc = kTotal + 1024;  // slack for manual 1024-B alignment
  static_assert(kAlloc <= 232448, "shared memory budget exceeded");
  static_assert(kB % 1024 == 0 && kStage % 1024 == 0, "SWIZZLE_128B tiles need 1024-B alignment");
  static_assert(DONE_RING > NS, "the producer looks NS tiles back in the ring of 'tile computed' barriers");
};

// K-major [rows][16] bf16 block (the folded bias and its "ones" partner): rows are exactly one 32-byte swizzle atom
// wide, 8-row groups are 256 B apart (SBO), LBO unused; layout type 6 = SWIZZLE_32B (16-byte chunk index XOR bit 2
// of the row).  The first version used the no-swizzle "interleave" layout, whose K = 16 MMA took ~500 cycles per tile
// instead of ~130 (DESIGN.md section 4.1).
LRB_DEVINL uint64_t umma_desc_k16_sw32(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3ffff) >> 4);
  d |= static_cast<uint64_t>(1) << 16;          // LBO (ignored)
  d |= static_cast<uint64_t>(256 >> 4) << 32;   // SBO
  d |= static_cast<uint64_t>(1) << 46;          // version
  d |= static_cast<uint64_t>(6) << 61;          // SWIZZLE_32B
  return d;
}

// Synchronisation (mbarriers; "tile" = one 256-item tile of one segment, counted per CTA in issue order):
//   full[s]        TMA bytes of shared-memory stage s have landed            producer -> MMA warp
//   done[t % 8][h] the MMAs of half-tile h of tile t have completed (one tcgen05.commit per half-tile):
//                  the accumulator stage (t & 1) * 2 + h is full            MMA -> epilogue warps (both CTAs of a pair)
//                  h == 1: AND shared-memory stage t % NS may be refilled    MMA -> TMA producer(s)
//   tmem_empty[a]  every epilogue warp has read accumulator stage a          epilogue -> MMA warp
// What bounds this kernel is the LATENCY of that loop, not a pipe (harness timeline, tools/tc_check with
// LRB_TIMELINE=1, DESIGN.md section 4.1): from "stage released" to "its next accumulator seen by the epilogue" pass
// ~1500 cycles of hand-offs (remote mbarrier arrivals of the pair's other CTA, the MMA warp's wake-up and issue, the
// commit's arrival) on top of the MMA itself; throughput = TMEM columns in flight / that cycle, hence four small
// stages instead of two large ones, and every hand-off kept as short as it goes.
template <int KMAX, int NS, bool kDense, int CG, int CMAX = MAX_C_SHARE_SMALL>
__global__ void __launch_bounds__(128 + EPI_WARPS * 32, 1)
score_topk_tc_kernel(const __grid_constant__ CUtensorMap tmap_a,
                     const __grid_constant__ CUtensorMap tmap_b,
                     const __grid_constant__ CUtensorMap tmap_bias, const ScoreParams p) {
  using L = SmemLayout<KMAX, NS, CG>;
  static_assert(CG == 1 || CG == 2, "cta_group is 1 or 2");
  constexpr int EPI_THREADS = EPI_WARPS * 32;
  constexpr int MAX_C_SHARE = CMAX;
  // CTA pair: cluster rank 0 leads (issues the MMAs, owns the barriers the pair synchronises on);
  // the pair walks the segments of "pair index" blockIdx.x / 2 and CTA `rank` owns user tile 2*m + rank.
  const uint32_t cta_rank = CG == 2 ? cluster_ctarank() : 0u;
  const int walk_id = CG == 2 ? static_cast<int>(blockIdx.x >> 1) : static_cast<int>(blockIdx.x);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>(
      (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));

  uint8_t* sA = smem + L::kA;
  uint8_t* sOnes = smem + L::kOnes;
  uint8_t* sB = smem + L::kB;
  float* sListS = reinterpret_cast<float*>(smem + L::kListS);
  int* sListI = reinterpret_cast<int*>(smem + L::kListI);
  int* sListN = reinterpret_cast<int*>(smem + L::kListN);
  int* sRowThr = reinterpret_cast<int*>(smem + L::kRowThr);          // [2][BM] double-buffered by segment parity
  volatile int* sSvc = reinterpret_cast<volatile int*>(smem + L::kRowThr + 2 * BM * 4);  // {cur_m, cur_seg, done}
  int* sExcl = reinterpret_cast<int*>(smem + L::kExcl);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::kBars);
  uint64_t* full_bar = bars;
  uint64_t* done_bar = bars + NS;
  uint64_t* tmem_empty_bar = bars + NS + 2 * DONE_RING;
  uint64_t* a_full_bar = bars + NS + 2 * DONE_RING + ACC_STAGES;
  uint64_t* a_empty_bar = a_full_bar + 1;
  uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(smem + L::kTmemPtr);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const bool has_bias = p.bias_blk != nullptr;

  // Programmatic dependent launch: the chunk launches of one lrb_score_topk call are independent (disjoint
  // users, disjoint scratch), so the next chunk's CTAs may take over SMs as soon as CTAs of this launch
  // exit instead of waiting for its slowest CTA.  (No-ops when launched without the attribute.)
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < NS; ++i) mbar_init(&full_bar[i], 1);
    for (int i = 0; i < 2 * DONE_RING; ++i) mbar_init(&done_bar[i], 1);
    // a stage is read by the 4 warps of one column part; pair: both CTAs' epilogues arrive on the leader's
    for (int i = 0; i < ACC_STAGES; ++i) mbar_init(&tmem_empty_bar[i], EPI_WARPS / PARTS * CG);
    mbar_init(a_full_bar, 1);
    mbar_init(a_empty_bar, 2);   // one commit from each MMA-issuing warp
    mbar_fence_init();
    sSvc[0] = -1; sSvc[1] = -1; sSvc[2] = 0; sSvc[3] = 0;
  }
  if (warp == 2) {
    if (CG == 2) {
      tmem_alloc_pair(tmem_ptr_s, TMEM_COLS);
      tmem_relinquish_pair();
    } else {
      tmem_alloc(tmem_ptr_s, TMEM_COLS);
      tmem_relinquish();
    }
  }
  if (warp == 3) {
    // "ones" block: column 0..2 = 1.0 (they multiply the hi/mid/lo bf16 terms of the bias)
    for (int i = lane; i < ONES_BYTES / 2; i += 32) {
      // 32-byte-swizzled K-major layout: element (row, k) at row*32 + ((k/8) ^ ((row/4)&1))*16 + (k%8)*2
      const int row = i >> 4;
      const int chunk = ((i >> 3) & 1) ^ ((row >> 2) & 1);   // logical K half stored in this physical chunk
      const int k = chunk * 8 + (i & 7);
      reinterpret_cast<__nv_bfloat16*>(sOnes)[i] = __float2bfloat16(k < 3 ? 1.0f : 0.0f);
    }
    // make the generic-proxy writes visible to the tensor core (async proxy)
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  tc_fence_before();
  if (CG == 2) cluster_sync_all();   // the peer's barriers must be initialised before anything remote arrives
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_s;

  // Register budget: the kernel is launched with 168 registers per thread (384 threads); the producer / MMA /
  // service warpgroup keeps 56 and hands the rest to the two epilogue warpgroups (224 each: two 64-register TMEM
  // load buffers plus the filter state).  128 * 56 + 256 * 224 = 64512 = 384 * 168.
  if (warp < 4) {
  setmaxnreg_dec<56>();
  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      SegmentWalk walk(p, walk_id);
      Segment sg;
      int stage = 0;
      uint32_t phase = 0;
      int seg_idx = 0;
      int t = 0;                      // tiles issued so far (all segments, scout tiles included)
      // bytes the (leader's) full barrier expects per stage: the parts of both CTAs
      const uint32_t stage_tx = (L::kBBytes + (has_bias ? L::kBiasBytes : 0)) * CG;
      const uint32_t a_full_lead = CG == 2 ? mapa_u32(smem_u32(a_full_bar), 0) : 0u;
      while (walk.next(sg)) {
        const int m_own = CG == 2 ? sg.m * 2 + static_cast<int>(cta_rank) : sg.m;
        if (seg_idx > 0) mbar_wait(a_empty_bar, (seg_idx - 1) & 1);
        if (CG == 2) {
          if (cta_rank == 0) mbar_expect_tx(a_full_bar, A_BYTES * 2);
          tma_load_2d_pair(sA, &tmap_a, a_full_lead, 0, m_own * BM);
        } else {
          mbar_expect_tx(a_full_bar, A_BYTES);
          tma_load_2d(sA, &tmap_a, a_full_bar, 0, m_own * BM);
        }
        const int n_scout = (kDense || p.scout_tiles <= 0) ? 0 : min(p.scout_tiles, sg.n1 - sg.n0);
        for (int it = -n_scout; it < sg.n1 - sg.n0; ++it, ++t) {
          const int n = it < 0 ? sg.n1 + it : sg.n0 + it;   // scout pass re-visits the segment's last tiles
          // stage t % NS was last read by the MMAs of tile t - NS
          if (t >= NS) mbar_wait(&done_bar[((t - NS) % DONE_RING) * 2 + 1], ((t - NS) / DONE_RING) & 1);
          uint8_t* st = sB + stage * L::kStage;
          if (CG == 2) {
            // each CTA fetches its 128 item rows (and its half of the bias block); all bytes are
            // accounted on the leader's barrier, which alone gates the pair's MMA
            if (cta_rank == 0) mbar_expect_tx(&full_bar[stage], stage_tx);
            const uint32_t full_lead = mapa_u32(smem_u32(&full_bar[stage]), 0);
            tma_load_2d_pair(st, &tmap_b, full_lead, 0, n * BN + static_cast<int>(cta_rank) * (BN / 2));
            if (has_bias)
              tma_load_2d_pair(st + L::kBBytes, &tmap_bias, full_lead, 0, n * BN + static_cast<int>(cta_rank) * (BN / 2));
          } else {
            mbar_expect_tx(&full_bar[stage], stage_tx);
            tma_load_2d(st, &tmap_b, &full_bar[stage], 0, n * BN);
            if (has_bias) tma_load_2d(st + B_BYTES, &tmap_bias, &full_bar[stage], 0, n * BN);
          }
          if (++stage == NS) { stage = 0; phase ^= 1; }
        }
        ++seg_idx;
      }
    }
  } else if (warp == 1 || warp == 2) {
    // ===================== MMA issuers =====================
    // TWO issuing warps, each with two of the four accumulator stages: warp 1 takes the even tiles, warp 2 the odd
    // ones; a tile is issued as two N = 128 half-tiles, each with its own stage and its own commit.  An issuing
    // thread is blocked in `tcgen05.mma` while the tensor pipe is busy and only then gets to its commit, its next
    // barrier waits and its descriptor arithmetic -- with a single issuer that gap (~150 cycles per tile) was idle
    // tensor-pipe time (MMA-only probe: 665-685 cycles per tile against 512 for back-to-back MMAs); with two, one
    // warp's gap hides behind the other's MMAs.  In each warp lane 0 polls "operands landed" and lane 1
    // "accumulator stage drained" with ONE try_wait instruction; lane 0 issues.
    if (cta_rank == 0) {
      constexpr uint32_t idesc = umma_idesc_bf16(BM * CG, HN);
      const int mw = warp - 1;        // this warp owns the accumulator stages 2*mw (first half-tile) and 2*mw+1
      SegmentWalk walk(p, walk_id);
      Segment sg;
      int seg_idx = 0;
      int t = 0;
      const uint64_t desc_a0 = umma_desc_k_sw128(smem_u32(sA));
      const uint64_t desc_ones = umma_desc_k16_sw32(smem_u32(sOnes));
      const uint32_t d_addr = tmem_base + static_cast<uint32_t>(mw * 2 * HN);
      // Half-tile h of a tile = item rows [h*64, h*64+64) of EACH CTA's 128-row part of the pair's tile (single CTAs:
      // rows [h*128, h*128+128) of the whole tile): offsets of the B operand / bias block inside a shared-memory stage
      constexpr uint32_t kHalfRows = HN / CG;
      constexpr uint32_t kHalfB = kHalfRows * BK * 2;        // bytes (whole SWIZZLE_128B atoms of 8 rows)
      constexpr uint32_t kHalfBias = kHalfRows * 32;         // bytes (whole SWIZZLE_32B atoms of 8 rows)
      while (walk.next(sg)) {
        if (lane == 0) mbar_wait(a_full_bar, seg_idx & 1);
        __syncwarp();
        const int n_scout = (kDense || p.scout_tiles <= 0) ? 0 : min(p.scout_tiles, sg.n1 - sg.n0);
        const int t_end = t + n_scout + (sg.n1 - sg.n0);
        for (t += (t & 1) ^ mw; t < t_end; t += 2) {   // this warp's tiles of the segment
          const int stage = t % NS;
          const uint32_t epar = static_cast<uint32_t>(((t >> 1) & 1) ^ 1);   // this warp's stages: used once per own tile
          // one lane, two waits in a row -- the accumulator stage (normally the later event) first.  (Two lanes
          // polling one barrier each in a single try_wait left ~450 cycles between the later lane's success and the
          // first MMA: harness timeline, A/B on B200 4.98 -> 4.78 ms at 4096 x 10M.)
          if (lane == 0) {
            mbar_wait(&tmem_empty_bar[2 * mw], epar);
            mbar_wait(&full_bar[stage], static_cast<uint32_t>((t / NS) & 1));
          }
          __syncwarp();
          if (lane == 0) {
            tc_fence_after();
            const uint32_t st = smem_u32(sB + stage * L::kStage);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              if (h == 1) {   // second accumulator stage of this tile
                mbar_wait(&tmem_empty_bar[2 * mw + 1], epar);
                tc_fence_after();
              }
              const uint64_t desc_b0 = umma_desc_k_sw128(st + h * kHalfB);
              const uint32_t d_h = d_addr + static_cast<uint32_t>(h * HN);
#pragma unroll
              for (int k = 0; k < BK / 16; ++k) {
                // advance 32 bytes (16 bf16) along K inside the 128-B swizzle atom: +2 in 16-B units
                if (CG == 2) umma_bf16_ss_pair(d_h, desc_a0 + 2 * k, desc_b0 + 2 * k, idesc, k > 0 ? 1u : 0u);
                else umma_bf16_ss(d_h, desc_a0 + 2 * k, desc_b0 + 2 * k, idesc, k > 0 ? 1u : 0u);
              }
              // folded bias: D += ones[128x16] * bias_blk[128x16]^T  (hi + mid + lo bf16 terms)
              if (has_bias) {
                const uint64_t desc_bias = umma_desc_k16_sw32(st + L::kBBytes + h * kHalfBias);
                if (CG == 2) umma_bf16_ss_pair(d_h, desc_ones, desc_bias, idesc, 1u);
                else umma_bf16_ss(d_h, desc_ones, desc_bias, idesc, 1u);
              }
              // one commit per half-tile: accumulator stage full (epilogues); the second one also means
              // "shared-memory stage free" (producers)
              if (CG == 2) umma_commit_pair(&done_bar[(t % DONE_RING) * 2 + h], 0b11);
              else umma_commit(&done_bar[(t % DONE_RING) * 2 + h]);
            }
          }
          __syncwarp();
        }
        t = t_end;
        if (lane == 0) {   // this warp's MMAs on the segment's user tile are done (the barrier counts both warps)
          if (CG == 2) umma_commit_pair(a_empty_bar, 0b11);
          else umma_commit(a_empty_bar);
        }
        __syncwarp();
        ++seg_idx;
      }
    }
  } else if (warp == 3) {
    // ===================== threshold service =====================
    // Background refresh of the per-row union bound: min over the row's stream slots of the published
    // c-th best scores (valid lower bound on the row's K-th best because c * slots >= K).  Written
    // into the threshold buffer of the segment it was computed for; a segment switch in between is
    // detected by re-reading the segment counter right before the write.
    if (!kDense && p.c_share > 0) {
      while (sSvc[2] == 0) {
        const int seg = sSvc[1];
        const int m = sSvc[0];
        if (seg >= 0) {
          for (int rr = lane; rr < BM; rr += 32) {
            const int b = m * BM + rr;
            if (b >= p.B) continue;
            const volatile int* gs = p.gslots + static_cast<size_t>(b) * p.gstride;
            int mn = INT_MAX;
            for (int sl = 0; sl < p.s_full; ++sl) {
#pragma unroll
              for (int pt = 0; pt < PARTS; ++pt) {
                const int v = gs[sl * PARTS + pt];
                mn = v < mn ? v : mn;
              }
            }
            if (mn > static_cast<int>(0x80808080) && sSvc[1] == seg) atomicMax(&sRowThr[(seg & 1) * BM + rr], mn);
          }
        }
        __nanosleep(2000);
      }
    }
  }
  } else {
    setmaxnreg_inc<224>();
    // ===================== epilogue =====================
    const int ew = warp - 4;          // 0..EPI_WARPS-1
    const int quad = ew & 3;          // TMEM lane quadrant == warp % 4
    const int part = ew >> 2;         // column part of the tile = the half-tile this warp reads
    const int et = ew * 32 + lane;    // epilogue thread index
    const int r = quad * 32 + lane;   // row inside the user tile
    const uint32_t ls = smem_u32(sListS + et);
    const uint32_t li = smem_u32(sListI + et);
    const uint32_t ln = smem_u32(sListN + et);

    SegmentWalk walk(p, walk_id);
    Segment sg;
    int t = 0;                        // tiles consumed so far (same count as the MMA warp's)
    int seg_idx = -1;
    // "accumulator stage drained": local barrier, or the leader's for a CTA pair
    const uint32_t acc_empty_addr0 = CG == 2 ? mapa_u32(smem_u32(&tmem_empty_bar[0]), 0) : smem_u32(&tmem_empty_bar[0]);
    const uint32_t peer_drain_addr =
        CG == 2 ? mapa_u32(smem_u32(const_cast<int*>(&sSvc[3])), cta_rank ^ 1u) : 0u;
    // Half-tile h of tile tt lives in accumulator stage (tt & 1) * 2 + h; this warp reads all 128 columns of half-tile
    // `part` as two 64-column BLOCKS q = 0, 1 (columns [q * 64, q * 64 + 64)).  Column c of half-tile h holds the item
    //     pair:   (c / 64) * 128 + h * 64 + c % 64   (columns 0..63 come from the leader CTA's item rows, 64..127 from the peer's)
    //     single: h * 128 + c
    // of the 256-item tile, i.e. block q is 64 consecutive items starting at item_off(q).
    constexpr int HCOLS = HN / 2;   // 64
    static_assert(HCOLS == 64, "one tcgen05.ld.32x32b.x64 per warp and block");
    const uint32_t taddr_quad = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
    auto half_taddr = [&](int tt, int q) {
      return taddr_quad + static_cast<uint32_t>(((tt & 1) * 2 + part) * HN + q * HCOLS);
    };
    auto item_off = [&](int q) { return CG == 2 ? q * 128 + part * 64 : part * 128 + q * 64; };
    // a warp waits for its half-tile before its first block and releases the accumulator stage after its second
    auto wait_half = [&](int tt) {   // the accumulator of half-tile `part` of tile tt is complete
      mbar_wait(&done_bar[(tt % DONE_RING) * 2 + part], (tt / DONE_RING) & 1);
      tc_fence_after();
    };
    auto release_half = [&](int tt) {   // this warp's loads of that accumulator stage have landed in its registers
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {            // (consecutive mbarriers are 8 bytes apart, in either address window)
        const uint32_t stg = static_cast<uint32_t>((tt & 1) * 2 + part);
        if (CG == 2) mbar_arrive_cluster(acc_empty_addr0 + stg * 8u);
        else mbar_arrive(&tmem_empty_bar[stg]);
      }
    };
    while (walk.next(sg)) {
      ++seg_idx;
      const int m_own = CG == 2 ? sg.m * 2 + static_cast<int>(cta_rank) : sg.m;
      const int b = m_own * BM + r;
      const bool live = b < p.B;
      int* rowthr = sRowThr + (seg_idx & 1) * BM;
      // per-segment state reset
      sts_s32(ln, 0);
      float own_thr = -INFINITY;
      int published = INT_MIN;
      if (part == 0) rowthr[r] = INT_MIN;
      const int my_slot = sg.slot * PARTS + part;
      const bool publishes = sg.slot < p.s_full;   // only full-stream threads feed the union bound
      const int* excl = nullptr;
      uint32_t bloom0 = 0u, bloom1 = 0u, bloom2 = 0u, bloom3 = 0u;
      if (!kDense && live && p.excl_sorted != nullptr) {
        excl = p.excl_sorted + static_cast<size_t>(b) * p.excl_stride;
        const uint4 bw = *reinterpret_cast<const uint4*>(p.excl_bloom + static_cast<size_t>(b) * 4);
        bloom0 = bw.x; bloom1 = bw.y; bloom2 = bw.z; bloom3 = bw.w;
      }
      uint32_t excl_s = 0u;
      if (!kDense && L::kExclSmem && p.excl_sorted != nullptr && p.excl_stride <= EX_CAP) {
        // stage the 128 rows' sorted exclusion lists in shared memory (binary-searched in the
        // lock-step compaction, where a global-memory search would stall the whole warp)
        const int total = BM * p.excl_stride;
        for (int i = et; i < total; i += EPI_THREADS) {
          const int rr = i / p.excl_stride;
          const int cc = i - rr * p.excl_stride;
          const int bb = m_own * BM + rr;
          sExcl[rr * EX_CAP + cc] =
              bb < p.B ? p.excl_sorted[static_cast<size_t>(bb) * p.excl_stride + cc] : INT_MAX;
        }
        excl_s = smem_u32(sExcl + r * EX_CAP);
      }
      asm volatile("bar.sync 1, %0;" ::"n"(EPI_THREADS));  // threshold buffer reset / sExcl visible
      if (et == 0) {
        sSvc[0] = m_own;
        __threadfence_block();
        sSvc[1] = seg_idx;      // the service warp starts refreshing this segment's buffer
      }
      int cnt = 0;   // records waiting in this thread's ring
      int drain_seen = sSvc[3];   // CTA-wide drain sequence number last honoured by this warp
      bool boot = !kDense;   // warp-uniform: without a scout pass the first tile of a segment always drains

      // ---------------- scout pass ----------------
      // The segment's last T0 tiles are scored once without any candidate handling: each thread only keeps
      // the m largest 16-item group maxima it sees (m = c + E, E = excluded ids inside the scouted id range,
      // so at least c of them belong to admissible items) and publishes the m-th.  The union bound is
      // therefore defined before the normal pass starts, which spares it the threshold-less first tiles.
      const int n_scout = (kDense || p.scout_tiles <= 0 || p.c_share <= 0) ? 0 : min(p.scout_tiles, sg.n1 - sg.n0);
      const int n_scout_run = (kDense || p.scout_tiles <= 0) ? 0 : min(p.scout_tiles, sg.n1 - sg.n0);
      if (n_scout_run > 0) {
        float tm[MAX_C_SHARE];   // the MAX_C_SHARE largest group maxima, descending
#pragma unroll
        for (int j = 0; j < MAX_C_SHARE; ++j) tm[j] = -INFINITY;
        for (int it = 0; it < n_scout_run; ++it, ++t) {
#pragma unroll 1
          for (int blk = 0; blk < 2; ++blk) {
            if (blk == 0) wait_half(t);
            // Columns past the end of the table (the ragged last tile) must not count as admissible items:
            // without a folded-bias block they score exactly 0 (TMA zero-fills out-of-bounds rows), and a
            // bound published from them could exceed a user's true K-th best.  valid = real items among
            // this thread's 64 columns of the block (warp-uniform; < 64 only in the last tile).
            const int valid = p.rows - ((sg.n1 - n_scout_run + it) * BN + item_off(blk));
            uint32_t w[64];
            tmem_ld_32x64(half_taddr(t, blk), w);
            tmem_ld_wait();
            if (blk == 1) release_half(t);
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              float q[16];
#pragma unroll
              for (int j = 0; j < 16; ++j) q[j] = __uint_as_float(w[g * 16 + j]);
              if (valid < HCOLS) {
#pragma unroll
                for (int j = 0; j < 16; ++j) q[j] = (g * 16 + j < valid) ? q[j] : -INFINITY;
              }
              const float m1 = max3(q[0], q[1], q[2]);
              const float m2 = max3(q[3], q[4], q[5]);
              const float m3 = max3(q[6], q[7], q[8]);
              const float m4 = max3(q[9], q[10], q[11]);
              const float m5 = max3(q[12], q[13], q[14]);
              float x = fmaxf(max3(m1, m2, m3), max3(m4, m5, q[15]));
#pragma unroll
              for (int j = 0; j < MAX_C_SHARE; ++j) {
                const float hi = fmaxf(tm[j], x);
                x = fminf(tm[j], x);
                tm[j] = hi;
              }
            }
          }
        }
        if (live && publishes && n_scout > 0) {
          // E = excluded ids that fall inside the scouted id range (any column part)
          int E = 0;
          if (excl != nullptr) {
            const int g_lo = p.row_offset + (sg.n1 - n_scout_run) * BN;
            const int g_hi = p.row_offset + sg.n1 * BN;
            int lo = 0, hi = p.excl_stride;
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (__ldg(excl + mid) < g_lo) lo = mid + 1; else hi = mid; }
            int lo2 = lo, hi2 = p.excl_stride;
            while (lo2 < hi2) { const int mid = (lo2 + hi2) >> 1; if (__ldg(excl + mid) < g_hi) lo2 = mid + 1; else hi2 = mid; }
            E = lo2 - lo;
          }
          const int mth = p.c_share + E;   // 1-based rank of the group maximum that is safe to publish
          float cb = -INFINITY;
#pragma unroll
          for (int j = 0; j < MAX_C_SHARE; ++j) cb = (mth == j + 1) ? tm[j] : cb;
          if (cb > -INFINITY) {
            published = float_to_key(cb);
            p.gslots[static_cast<size_t>(b) * p.gstride + my_slot] = published;
          }
        }
        boot = false;
        // give the threshold service a bounded moment to pick the bound up (never blocks on other CTAs)
#pragma unroll 1
        for (int spin = 0; spin < 40; ++spin) {
          const int kk = *reinterpret_cast<volatile int*>(rowthr + r);
          if (__all_sync(0xffffffffu, kk != INT_MIN || !live)) break;
          __nanosleep(250);
        }
      }
      float4* ring = reinterpret_cast<float4*>(
          p.ring + (static_cast<size_t>(blockIdx.x) * EPI_THREADS + et) * (RING_GROUPS * RING_REC_BYTES));
      const int limit_gid = p.row_offset + p.rows;

      // lock-step drain of the warp's rings + publication of the improved bounds (out of line, state in local memory)
      DrainState dst;
      dst.ring = ring; dst.excl = excl; dst.rowthr = rowthr + r;
      dst.gslot = (live && p.c_share > 0 && publishes) ? p.gslots + static_cast<size_t>(b) * p.gstride + my_slot : nullptr;
      dst.excl_s = excl_s; dst.bloom0 = bloom0; dst.bloom1 = bloom1; dst.bloom2 = bloom2; dst.bloom3 = bloom3;
      dst.ls = ls; dst.li = li; dst.ln = ln;
      dst.excl_stride = p.excl_stride; dst.K = p.K; dst.limit_gid = limit_gid; dst.c_share = p.c_share;
      dst.published = published; dst.live = live;
      auto drain = [&]() {
        own_thr = drain_rings<EPI_THREADS, KMAX, CMAX>(&dst, cnt, own_thr);
        cnt = 0;
      };

      const uint32_t rowthr_s = smem_u32(rowthr + r);
      const uint32_t drain_seq_s = smem_u32(const_cast<int*>(&sSvc[3]));

      if (kDense) {
        for (int n = sg.n0; n < sg.n1; ++n, ++t) {
#pragma unroll 1
          for (int blk = 0; blk < 2; ++blk) {
            if (blk == 0) wait_half(t);
            uint32_t v[64];
            tmem_ld_32x64(half_taddr(t, blk), v);
            tmem_ld_wait();
            if (blk == 1) release_half(t);
            const int row = m_own * BM + r;
            const int col0 = n * BN + item_off(blk);
            if (row < p.B) {
              float* dstp = p.dense_out + static_cast<size_t>(row) * p.dense_ld + col0;
              if (col0 + HCOLS <= p.rows && (p.dense_ld & 3) == 0) {
#pragma unroll
                for (int j = 0; j < HCOLS / 4; ++j)
                  reinterpret_cast<float4*>(dstp)[j] =
                      make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                                  __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
              } else {
#pragma unroll
                for (int j = 0; j < HCOLS; ++j)
                  if (col0 + j < p.rows) dstp[j] = __uint_as_float(v[j]);
              }
            }
          }
        }
      } else {
        // ---------------- the filter loop ----------------
        // Per half-tile a thread's 64 columns arrive as one 64-register load (tcgen05.ld.32x32b.x64); the stage goes
        // back to the MMA warp as soon as the load has landed, before anything is computed.  The two half-tiles of a
        // tile use separate buffers so that the second load may be in flight while the first half is reduced (the
        // register budget for this comes from setmaxnreg, see the role dispatch).
        // Per half: four 16-column FMNMX3 trees -> four group maxima -> ONE compare and ONE (rarely taken) branch;
        // a group whose maximum reaches the thread's threshold is not inspected, it is dumped into the thread's
        // ring (5 stores).  Everything else that used to be decided per tile -- ring occupancy, the CTA-wide drain
        // sequence, the bootstrap drain -- sits behind one warp-uniform branch that is only taken when some lane had
        // a hit or the drain sequence moved.  (ncu, round 2: the nine branches per tile of the previous loop cost
        // ~30 % of the epilogue's cycles in branch-resolution stalls.)
        auto group_max = [](const uint32_t (&x)[64], int o) -> float {
          const float m1 = max3(__uint_as_float(x[o + 0]), __uint_as_float(x[o + 1]), __uint_as_float(x[o + 2]));
          const float m2 = max3(__uint_as_float(x[o + 3]), __uint_as_float(x[o + 4]), __uint_as_float(x[o + 5]));
          const float m3 = max3(__uint_as_float(x[o + 6]), __uint_as_float(x[o + 7]), __uint_as_float(x[o + 8]));
          const float m4 = max3(__uint_as_float(x[o + 9]), __uint_as_float(x[o + 10]), __uint_as_float(x[o + 11]));
          const float m5 = max3(__uint_as_float(x[o + 12]), __uint_as_float(x[o + 13]), __uint_as_float(x[o + 14]));
          return fmaxf(max3(m1, m2, m3), max3(m4, m5, __uint_as_float(x[o + 15])));
        };
        auto dump_half = [&](const uint32_t (&x)[64], const float (&g)[4], float t_eff, int gid0) {
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            if (g[q] >= t_eff) {
              float4* rec = ring + cnt * (RING_REC_BYTES / 16);
#pragma unroll
              for (int j = 0; j < 4; ++j)
                rec[j] = make_float4(__uint_as_float(x[q * 16 + 4 * j]), __uint_as_float(x[q * 16 + 4 * j + 1]),
                                     __uint_as_float(x[q * 16 + 4 * j + 2]), __uint_as_float(x[q * 16 + 4 * j + 3]));
              reinterpret_cast<int*>(rec + 4)[0] = gid0 + q * 16;
              ++cnt;
            }
          }
        };
        if (!live) own_thr = INFINITY;   // rows beyond B never produce candidates
        uint32_t va[64], vb[64];
#pragma unroll 1
        for (int n = sg.n0; n < sg.n1; ++n, ++t) {
          // the row's shared threshold and the CTA's drain sequence: shared-space loads issued ahead of the waits.
          // key_to_float(INT_MIN) is a NaN, which fmaxf ignores: an unset shared threshold leaves own_thr.
          const int kk = lds_volatile_s32(rowthr_s);
          const int seq0 = lds_volatile_s32(drain_seq_s);
          const float t_eff = fmaxf(own_thr, key_to_float(kk));
          const int tile_gid0 = p.row_offset + n * BN;

          wait_half(t);
          tmem_ld_32x64(half_taddr(t, 0), va);
          tmem_ld_32x64(half_taddr(t, 1), vb);     // in flight while the first block is reduced
          float ga[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) ga[q] = group_max(va, q * 16);
          const bool hit_a = fmaxf(fmaxf(ga[0], ga[1]), fmaxf(ga[2], ga[3])) >= t_eff;
          if (__builtin_expect(hit_a, 0)) dump_half(va, ga, t_eff, tile_gid0 + item_off(0));

          tmem_ld_wait();
          release_half(t);
          float gb[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) gb[q] = group_max(vb, q * 16);
          const bool hit_b = fmaxf(fmaxf(gb[0], gb[1]), fmaxf(gb[2], gb[3])) >= t_eff;
          if (__builtin_expect(hit_b, 0)) dump_half(vb, gb, t_eff, tile_gid0 + item_off(1));

          if (__builtin_expect(__any_sync(0xffffffffu, hit_a || hit_b || boot || seq0 != drain_seen), 0)) {
            // uniform point: a tile adds at most 8 records per thread, so draining whenever some lane
            // holds more than RING_GROUPS-8 keeps every ring within capacity.  The first tile of a segment without
            // a scout pass always drains (bootstrap): every stream then holds K entries and publishes its c-th best
            // within the first microseconds, which defines the union bound.  Drains are synchronised across the
            // CTA's epilogue warps: a warp that must drain bumps a shared sequence number and every warp drains at
            // its next tile boundary.  A drain stalls the accumulator ring for everybody, so simultaneous
            // drains cost one stall, not one per warp.
            const bool need = __any_sync(0xffffffffu, cnt > RING_GROUPS - 8 || (boot && cnt > 0));
            int seq = lds_volatile_s32(drain_seq_s);
            if (need && seq == drain_seen) {
              if (lane == 0) {
                atomicAdd(const_cast<int*>(&sSvc[3]), 1);
                // a drain stalls the pair's accumulator ring: let the peer CTA drain at the same time
                if (CG == 2) red_add_cluster_u32(peer_drain_addr, 1u);
              }
              seq += 1;
            }
            if (need || seq != drain_seen) {
              drain_seen = lds_volatile_s32(drain_seq_s);
              boot = false;
              drain();
            }
          }
        }
      }

      if (!kDense) drain();   // final drain of this segment (whole warp, lock-step)

      if (!kDense && live) {
        const int held = lds_s32(ln);
        const size_t base = (static_cast<size_t>(b) * p.slots + my_slot);
        p.part_cnt[base] = held;
        for (int i = 0; i < held; ++i) {
          p.part_scores[base * p.K + i] = lds_f32(ls + i * EPI_THREADS * 4);
          p.part_ids[base * p.K + i] = lds_s32(li + i * EPI_THREADS * 4);
        }
      }
      asm volatile("bar.sync 1, %0;" ::"n"(EPI_THREADS));  // before the next segment resets its buffer
    }
    if (et == 0) sSvc[2] = 1;   // all segments of this CTA are done: stop the threshold service
  }

  // ... but no launch may COMPLETE before its predecessor has: what follows the last chunk in the stream
  // (the merge kernel) must see the results of every chunk.
  asm volatile("griddepcontrol.wait;" ::: "memory");
  tc_fence_before();
  if (CG == 2) cluster_sync_all();   // the peer may still read this CTA's tile halves / arrive on its barriers
  else __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    if (CG == 2) tmem_dealloc_pair(tmem_base, TMEM_COLS);
    else tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

}  // namespace tc
}  // namespace lrb
