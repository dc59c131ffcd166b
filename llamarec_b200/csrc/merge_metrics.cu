// k-way merge of per-split / per-rank candidate sets + Recall/MRR/NDCG + candidate emission,
// one fused kernel (north_star subsystem 3).
//
// Replaces, per user,
//   rank = (-scores).argsort(dim=1)            trainer/utils.py:56   (full sort of N+1 scores)
//   hits / Recall / MRR / NDCG @ ks            trainer/utils.py:61-88
//   torch.topk(scores, 20) + `label in top20`  trainer/lru.py:82-88, 124-132
// by a selection over the <= n_lists*K_in candidates the scoring kernel kept: the label's rank in
// the merged list is its rank in the full catalogue whenever that rank is < K_out, which is all
// the metrics at k <= K_out need.
//
// One warp per user.  Entries live in registers (up to 16 per lane) or, for very wide fan-in
// (tiny batches split over many CTAs), are re-read from global memory each round.
#include "api_util.h"
#include "common.cuh"

#include <climits>

namespace lrb {
namespace mm {

constexpr int WARPS = 8;
constexpr int MAX_PER_LANE = 32;   // register-resident entries per lane (up to 1024 per user); the kernel is
                                   // instantiated for 2/4/8/16/32 so that narrow fan-in does not pay for 32.
                                   // (Beyond that every round re-reads the lists from global memory: the 19 x 50
                                   // candidates per user of the exact-fp32 path at C3 took 494 us that way.)
constexpr int MAX_KS = 8;
constexpr int MAX_DST = 16;    // scatter mode: destination buffers (ranks of one node)

struct Params {
  const float* list_scores;
  const int* list_ids;
  const int* list_cnt;         // may be null
  int n_lists;
  long long stride_list, stride_user, cnt_stride_list, cnt_stride_user;
  int K_in, B, K_out;
  const long long* labels;     // may be null
  int ks[MAX_KS];
  int n_ks;
  float* top_scores;           // [B][K_out], rows out_stride elements apart
  int* top_ids;                // [B][K_out], rows out_stride elements apart
  long long out_stride;
  // scatter mode (users_per_dst > 0): user b's list goes to row (b % users_per_dst) of destination
  // b / users_per_dst -- the recv buffer of the rank that owns the user, written over NVLink; this is the
  // all-to-all of the row-sharded retrieval step fused into the merge that produces its payload.
  float* dst_scores[MAX_DST];
  int* dst_ids[MAX_DST];
  int users_per_dst;
  int* label_rank;             // [B] (may be null)
  float* metric_sums;          // [3*n_ks] (may be null)
};

struct Best {
  float s;
  int id;
  int lane;
};

LRB_DEVINL Best warp_best(float s, int id, int lane) {
  Best b{s, id, lane};
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float os = __shfl_xor_sync(0xffffffffu, b.s, o);
    const int oi = __shfl_xor_sync(0xffffffffu, b.id, o);
    const int ol = __shfl_xor_sync(0xffffffffu, b.lane, o);
    if (better(os, oi, b.s, b.id) || (os == b.s && oi == b.id && ol < b.lane)) {
      b.s = os; b.id = oi; b.lane = ol;
    }
  }
  return b;
}

template <int PER_LANE>
__global__ void __launch_bounds__(WARPS * 32) merge_metrics_kernel(const Params p) {
  __shared__ float s_sums[WARPS][3 * MAX_KS];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * WARPS + warp;
  float acc[3 * MAX_KS];
#pragma unroll
  for (int i = 0; i < 3 * MAX_KS; ++i) acc[i] = 0.f;

  if (b < p.B) {
    const float* sc = p.list_scores + static_cast<size_t>(b) * p.stride_user;
    const int* id = p.list_ids + static_cast<size_t>(b) * p.stride_user;
    const int total_slots = p.n_lists * p.K_in;
    const bool in_regs = total_slots <= 32 * PER_LANE;
    float* out_s = p.top_scores + static_cast<size_t>(b) * p.out_stride;
    int* out_i = p.top_ids + static_cast<size_t>(b) * p.out_stride;
    if (p.users_per_dst > 0) {
      const int d = b / p.users_per_dst;
      const size_t row = static_cast<size_t>(b - d * p.users_per_dst);
      out_s = p.dst_scores[d] + row * p.out_stride;
      out_i = p.dst_ids[d] + row * p.out_stride;
    }
    int my_rank = -1;
    const long long label = p.labels ? p.labels[b] : -1;
    // One list that is already sorted -- strictly by (score key desc, id asc), every entry finite or +inf -- is its
    // own merge (the one list per user of the select paths): one warp pass checks it and it is copied instead of
    // running K_out selection rounds.  Same output as the rounds.
    bool copied = false;
    if (p.n_lists == 1) {
      int cnt = p.list_cnt ? p.list_cnt[static_cast<size_t>(b) * p.cnt_stride_user] : p.K_in;
      cnt = cnt < p.K_in ? cnt : p.K_in;
      bool ok = true;
      for (int i = lane; i < cnt; i += 32) {
        const float s = sc[i];
        const int d = id[i];
        const int k = float_to_key(s);
        ok = ok && s > -INFINITY && d != INT_MAX;      // (false for NaN too)
        if (i + 1 < cnt) {
          const int k1 = float_to_key(sc[i + 1]);
          ok = ok && (k > k1 || (k == k1 && d < id[i + 1]));
        }
      }
      copied = __all_sync(0xffffffffu, ok);
      if (copied) {
        for (int k = lane; k < p.K_out; k += 32) {
          const bool v = k < cnt;
          const int d = v ? id[k] : -1;
          out_s[k] = v ? sc[k] : -INFINITY;
          out_i[k] = d;
          const unsigned hit = __ballot_sync(__activemask(), v && static_cast<long long>(d) == label);
          if (my_rank < 0 && hit) my_rank = (k - lane) + __ffs(hit) - 1;
        }
        my_rank = __reduce_max_sync(0xffffffffu, my_rank);
      }
    }
    if (!copied) {

    float es[PER_LANE];
    int ei[PER_LANE];
    if (in_regs) {
#pragma unroll
      for (int q = 0; q < PER_LANE; ++q) {
        const int e = q * 32 + lane;
        es[q] = -INFINITY;
        ei[q] = INT_MAX;
        if (e < total_slots) {
          const int l = e / p.K_in;
          const int i = e - l * p.K_in;
          const int cnt = p.list_cnt ? p.list_cnt[b * p.cnt_stride_user + l * p.cnt_stride_list] : p.K_in;
          if (i < cnt) {
            es[q] = sc[l * p.stride_list + i];
            ei[q] = id[l * p.stride_list + i];
          }
        }
      }
    }

    // floor for the global-memory path: entries must be strictly "after" the previous winner
    float prev_s = INFINITY;
    int prev_id = -1;
    // the merged list is collected in registers (lane k % 32 holds entry k) and written once at the end: two
    // coalesced stores per user instead of 2 * K_out four-byte stores by lane 0 -- in scatter mode those are remote
    // stores over NVLink (8-GPU step: 132 us for 32768 users before this change)
    float res_s[2] = {-INFINITY, -INFINITY};
    int res_i[2] = {-1, -1};
    float wide_s = -INFINITY;
    int wide_i = -1;
    for (int k = 0; k < p.K_out; ++k) {
      float w_s;
      int w_id;
      if (in_regs) {
        // lane-local best score (max tree), warp-wide maximum by one redux on the order-preserving key
        float bs = es[0];
#pragma unroll
        for (int q = 1; q + 1 < PER_LANE; q += 2) bs = max3(bs, es[q], es[q + 1]);
        bs = fmaxf(bs, es[PER_LANE - 1]);
        const int key = float_to_key(bs);
        const int wkey = __reduce_max_sync(0xffffffffu, key);
        const bool mine = key == wkey;
        // among this lane's entries that carry the winning score: lowest id, and how many there are
        int bi = INT_MAX, n_eq = 0;
#pragma unroll
        for (int q = 0; q < PER_LANE; ++q) {
          const bool eq = mine && es[q] == bs;
          bi = (eq && ei[q] < bi) ? ei[q] : bi;
          n_eq += eq ? 1 : 0;
        }
        // ties across lanes (or inside one) resolve towards the lowest id
        w_id = __reduce_min_sync(0xffffffffu, mine ? bi : INT_MAX);
        w_s = key_to_float(wkey);
        if (wkey == float_to_key(-INFINITY)) { w_id = INT_MAX; w_s = -INFINITY; }
        (void)n_eq;
        // the owner of (w_s, w_id) retires that entry (first match only, so duplicates stay countable)
        bool done = !(mine && bi == w_id) || w_id == INT_MAX;
#pragma unroll
        for (int q = 0; q < PER_LANE; ++q) {
          const bool hit = !done && es[q] == w_s && ei[q] == w_id;
          es[q] = hit ? -INFINITY : es[q];
          ei[q] = hit ? INT_MAX : ei[q];
          done = done || hit;
        }
      } else {
        float bs = -INFINITY;
        int bi = INT_MAX;
        for (int e = lane; e < total_slots; e += 32) {
          const int l = e / p.K_in;
          const int i = e - l * p.K_in;
          const int cnt = p.list_cnt ? p.list_cnt[b * p.cnt_stride_user + l * p.cnt_stride_list] : p.K_in;
          if (i >= cnt) continue;
          const float s = sc[l * p.stride_list + i];
          const int d = id[l * p.stride_list + i];
          // skip everything already emitted: strictly after (prev_s, prev_id) in the total order
          if (!(better(prev_s, prev_id, s, d))) continue;
          if (better(s, d, bs, bi)) { bs = s; bi = d; }
        }
        const Best w = warp_best(bs, bi, lane);
        w_s = w.s;
        w_id = w.id;
      }
      prev_s = w_s;
      prev_id = w_id;
      const bool valid = w_id != INT_MAX;
      if (lane == (k & 31)) {
        if (k < 32) { res_s[0] = valid ? w_s : -INFINITY; res_i[0] = valid ? w_id : -1; }
        else if (k < 64) { res_s[1] = valid ? w_s : -INFINITY; res_i[1] = valid ? w_id : -1; }
      }
      if (k >= 64) {   // wide lists (K_out > 64): entries staged per group of 32, one coalesced store per group
        if (lane == (k & 31)) { wide_s = valid ? w_s : -INFINITY; wide_i = valid ? w_id : -1; }
        if ((k & 31) == 31 || k == p.K_out - 1) {
          const int g = k & ~31;
          if (g + lane <= k) { out_s[g + lane] = wide_s; out_i[g + lane] = wide_i; }
        }
      }
      if (valid && my_rank < 0 && static_cast<long long>(w_id) == label) my_rank = k;
    }
    if (lane < p.K_out) { out_s[lane] = res_s[0]; out_i[lane] = res_i[0]; }
    if (lane + 32 < p.K_out) { out_s[lane + 32] = res_s[1]; out_i[lane + 32] = res_i[1]; }
    }
    if (p.label_rank && lane == 0) p.label_rank[b] = my_rank;
    if (p.labels && my_rank >= 0 && lane == 0) {
      // one relevant item per user: Recall@k = [r<k], MRR@k = [r<k]/(r+1), NDCG@k = [r<k]/log2(r+2)
      // (trainer/utils.py:61-88 with answer_count == 1, hence idcg == 1)
      const float mrr = 1.0f / static_cast<float>(my_rank + 1);
      const float ndcg = 1.0f / log2f(static_cast<float>(my_rank + 2));
#pragma unroll
      for (int i = 0; i < MAX_KS; ++i) {
        if (i < p.n_ks && my_rank < p.ks[i]) {
          acc[3 * i + 0] = 1.0f;
          acc[3 * i + 1] = mrr;
          acc[3 * i + 2] = ndcg;
        }
      }
    }
  }
  if (p.metric_sums != nullptr) {
    if (lane == 0) {
#pragma unroll
      for (int i = 0; i < 3 * MAX_KS; ++i) s_sums[warp][i] = acc[i];
    }
    __syncthreads();
    if (threadIdx.x < 3 * p.n_ks) {
      float t = 0.f;
      for (int w = 0; w < WARPS; ++w) t += s_sums[w][threadIdx.x];
      if (t != 0.f) atomicAdd(p.metric_sums + threadIdx.x, t);
    }
  }
}

}  // namespace mm
}  // namespace lrb

namespace {
int merge_launch(const float* list_scores, const int32_t* list_ids, const int32_t* list_cnt, int n_lists,
                 int64_t stride_list, int64_t stride_user, int64_t cnt_stride_list, int64_t cnt_stride_user,
                 int K_in, int B, int K_out, const int64_t* labels, const int32_t* ks_host, int n_ks,
                 float* top_scores, int32_t* top_ids, float* const* dst_scores_host,
                 int32_t* const* dst_ids_host, int n_dst, int users_per_dst, int64_t out_stride,
                 int32_t* label_rank, float* metric_sums, void* stream) {
  using namespace lrb;
  int rc = check_arch();
  if (rc != LRB_OK) return rc;
  LRB_REQUIRE(list_scores && list_ids, "lrb_merge_metrics: null pointer");
  LRB_REQUIRE(n_lists >= 1 && K_in >= 1 && B >= 1 && K_out >= 1, "lrb_merge_metrics: bad shape");
  LRB_REQUIRE(n_ks >= 0 && n_ks <= mm::MAX_KS, "lrb_merge_metrics: at most %d cut-offs", mm::MAX_KS);
  LRB_REQUIRE(n_ks == 0 || ks_host != nullptr, "lrb_merge_metrics: ks missing");
  LRB_REQUIRE(out_stride == 0 || out_stride >= K_out, "lrb_merge_metrics: out_stride must be 0 or >= K_out");
  mm::Params p = {};
  p.list_scores = list_scores; p.list_ids = list_ids; p.list_cnt = list_cnt; p.n_lists = n_lists;
  p.stride_list = stride_list; p.stride_user = stride_user;
  p.cnt_stride_list = cnt_stride_list; p.cnt_stride_user = cnt_stride_user;
  p.K_in = K_in; p.B = B; p.K_out = K_out;
  p.labels = reinterpret_cast<const long long*>(labels);
  for (int i = 0; i < mm::MAX_KS; ++i) p.ks[i] = i < n_ks ? ks_host[i] : 0;
  p.n_ks = labels ? n_ks : 0;
  p.top_scores = top_scores; p.top_ids = top_ids; p.label_rank = label_rank;
  p.out_stride = out_stride > 0 ? out_stride : K_out;
  p.users_per_dst = 0;
  if (n_dst > 0) {
    LRB_REQUIRE(n_dst <= mm::MAX_DST && users_per_dst >= 1 && dst_scores_host && dst_ids_host,
                "lrb_merge_metrics_scatter: 1..%d destinations with users_per_dst >= 1", mm::MAX_DST);
    LRB_REQUIRE(static_cast<long long>(n_dst) * users_per_dst >= B,
                "lrb_merge_metrics_scatter: %d destinations x %d users do not cover B=%d", n_dst, users_per_dst, B);
    for (int d = 0; d < n_dst; ++d) {
      LRB_REQUIRE(dst_scores_host[d] && dst_ids_host[d], "lrb_merge_metrics_scatter: null destination %d", d);
      p.dst_scores[d] = dst_scores_host[d];
      p.dst_ids[d] = dst_ids_host[d];
    }
    p.users_per_dst = users_per_dst;
  } else {
    LRB_REQUIRE(top_scores && top_ids, "lrb_merge_metrics: null output pointer");
  }
  p.metric_sums = (labels && n_ks > 0) ? metric_sums : nullptr;
  const int grid = (B + mm::WARPS - 1) / mm::WARPS;
  const long long total = static_cast<long long>(n_lists) * K_in;
  cudaStream_t st = as_stream(stream);
  if (total <= 64) mm::merge_metrics_kernel<2><<<grid, mm::WARPS * 32, 0, st>>>(p);
  else if (total <= 128) mm::merge_metrics_kernel<4><<<grid, mm::WARPS * 32, 0, st>>>(p);
  else if (total <= 256) mm::merge_metrics_kernel<8><<<grid, mm::WARPS * 32, 0, st>>>(p);
  else if (total <= 512) mm::merge_metrics_kernel<16><<<grid, mm::WARPS * 32, 0, st>>>(p);
  else mm::merge_metrics_kernel<mm::MAX_PER_LANE><<<grid, mm::WARPS * 32, 0, st>>>(p);
  LRB_CUDA_TRY(cudaGetLastError());
  return LRB_OK;
}
}  // namespace

extern "C" int lrb_merge_metrics(const float* list_scores, const int32_t* list_ids, const int32_t* list_cnt,
                                 int n_lists, int64_t stride_list, int64_t stride_user,
                                 int64_t cnt_stride_list, int64_t cnt_stride_user, int K_in, int B, int K_out,
                                 const int64_t* labels, const int32_t* ks_host, int n_ks, float* top_scores,
                                 int32_t* top_ids, int64_t out_stride, int32_t* label_rank, float* metric_sums,
                                 void* stream) {
  return merge_launch(list_scores, list_ids, list_cnt, n_lists, stride_list, stride_user, cnt_stride_list,
                      cnt_stride_user, K_in, B, K_out, labels, ks_host, n_ks, top_scores, top_ids, nullptr, nullptr,
                      0, 0, out_stride, label_rank, metric_sums, stream);
}

extern "C" int lrb_merge_metrics_scatter(const float* list_scores, const int32_t* list_ids,
                                         const int32_t* list_cnt, int n_lists, int64_t stride_list,
                                         int64_t stride_user, int64_t cnt_stride_list, int64_t cnt_stride_user,
                                         int K_in, int B, int K_out, float* const* dst_scores_host,
                                         int32_t* const* dst_ids_host, int n_dst, int users_per_dst,
                                         int64_t out_stride, void* stream) {
  return merge_launch(list_scores, list_ids, list_cnt, n_lists, stride_list, stride_user, cnt_stride_list,
                      cnt_stride_user, K_in, B, K_out, nullptr, nullptr, 0, nullptr, nullptr, dst_scores_host,
                      dst_ids_host, n_dst, users_per_dst, out_stride, nullptr, nullptr, stream);
}
