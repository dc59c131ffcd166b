// Exact fp32 top-K on large catalogues (LRURec.retrieve(precision="exact")): the bf16 tensor-core candidates are
// rescored with the fp32 path's own arithmetic, and a per-user bound eps_u on |bf16 score - fp32 score| either
// certifies the rescored list or gives a threshold below which no item of the fp32 top K can lie.
//   lrb_exact_rescore   pass A: rescore the bf16 top-K' list, certify it or emit the collect threshold
//   lrb_score_collect   pass B (score.cu): every item whose bf16 score reaches the threshold
//   lrb_exact_select    exact top K over the collected ids
// DESIGN.md section 2.1 derives the bound.
#include "api_util.h"
#include "common.cuh"

#include <climits>
#include <cmath>

namespace lrb {
namespace exact {

constexpr int WARPS = 8;   // one warp per user
constexpr int D = 64;

// eps_u = RHO * S_u + RHO_B * b_max + FLOOR, S_u = sum_i |u_i| * c_i (DESIGN.md section 2.1)
constexpr float RHO = 0x1p-7f + 0x1p-12f;
constexpr float RHO_B = 0x1p-12f;
constexpr float FLOOR = 0x1p-96f;
// larger bounds go to the fp32 path: |score| <= S_u + b_max stays far from the fp32 overflow threshold
constexpr float EPS_MAX = 0x1p100f;

// The fp32 path's score (score.cu, score_f32_kernel), operation for operation: four interleaved 16-FMA chains,
// ((a0 + a1) + (a2 + a3)) + bias.  u is the user's state in shared memory, `local` the shard-local row.
LRB_DEVINL float score_f32(const float* u, const float* table, const float* bias_pad, int local) {
  const float4* e4 = reinterpret_cast<const float4*>(table + static_cast<size_t>(local) * D);
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
  for (int k4 = 0; k4 < D / 4; ++k4) {
    const float4 ev = __ldg(e4 + k4);
    a0 = fmaf(u[4 * k4 + 0], ev.x, a0);
    a1 = fmaf(u[4 * k4 + 1], ev.y, a1);
    a2 = fmaf(u[4 * k4 + 2], ev.z, a2);
    a3 = fmaf(u[4 * k4 + 3], ev.w, a3);
  }
  return ((a0 + a1) + (a2 + a3)) + __ldg(bias_pad + local);
}

LRB_DEVINL bool finite(float x) { return fabsf(x) <= 3.402823466e38f; }

struct RescoreParams {
  const float* u;            // [B][64] fp32 user states
  const float* table;        // [rows][64] fp32 shard rows
  const float* bias_pad;     // shard bias (lrb_prepare_table)
  const float* bound;        // [65]: c_i = max_j |table[j][i]|, then b_max
  int B, rows, row_offset;
  const float* cand_scores;  // [B][Kc] bf16 candidate list, sorted (score desc, id asc); missing entries id < 0
  const int* cand_ids;
  int Kc, K;
  float* out_scores;         // [B][K]
  int* out_ids;
  int* out_cnt;              // [B]
  int8_t* path;              // [B]
  float* tau;                // [B]
  float* fk;                 // [B]
};

__global__ void __launch_bounds__(WARPS * 32) exact_rescore_kernel(const RescoreParams p) {
  __shared__ float s_u[WARPS][D];
  __shared__ float s_sc[WARPS][64];
  __shared__ int s_id[WARPS][64];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * WARPS + warp;
  if (b >= p.B) return;                         // (no block-level barrier below)
  const float u0 = p.u[static_cast<size_t>(b) * D + lane];
  const float u1 = p.u[static_cast<size_t>(b) * D + lane + 32];
  s_u[warp][lane] = u0;
  s_u[warp][lane + 32] = u1;
  // eps_u with every operation rounded upwards: the computed value is >= the bound's exact value
  float S = __fadd_ru(__fmul_ru(fabsf(u0), p.bound[lane]), __fmul_ru(fabsf(u1), p.bound[lane + 32]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) S = __fadd_ru(S, __shfl_xor_sync(0xffffffffu, S, o));
  const float eps = __fmaf_ru(RHO, S, __fmaf_ru(RHO_B, p.bound[D], FLOOR));
  __syncwarp();

  bool bad = !(eps <= EPS_MAX);                 // NaN too
  int n_real = 0;
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const int e = lane + 32 * q;
    const int id = e < p.Kc ? p.cand_ids[static_cast<size_t>(b) * p.Kc + e] : -1;
    const long long local = static_cast<long long>(id) - p.row_offset;
    const bool valid = id >= 0 && local >= 0 && local < p.rows;
    const float sc = valid ? score_f32(s_u[warp], p.table, p.bias_pad, static_cast<int>(local)) : -INFINITY;
    bad = bad || (valid && !finite(sc));
    s_sc[warp][e] = sc;
    s_id[warp][e] = valid ? id : INT_MAX;
    n_real += __popc(__ballot_sync(0xffffffffu, valid));
  }
  bad = __any_sync(0xffffffffu, bad);
  __syncwarp();

  // rank sort of the rescored list into (score desc, id asc)
  int rank[2];
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const int e = lane + 32 * q;
    const float sc = s_sc[warp][e];
    const int id = s_id[warp][e];
    int r = 0;
    for (int j = 0; j < p.Kc; ++j) {
      const int ij = s_id[warp][j];
      r += (ij != INT_MAX && better(s_sc[warp][j], ij, sc, id)) ? 1 : 0;
    }
    rank[q] = (e < p.Kc && id != INT_MAX) ? r : INT_MAX;
  }
  // f_K: the K-th best rescored score (-inf when the list holds fewer than K entries)
  float f_k = -INFINITY;
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const unsigned hit = __ballot_sync(0xffffffffu, rank[q] == p.K - 1);
    if (hit) f_k = __shfl_sync(0xffffffffu, s_sc[warp][lane + 32 * q], __ffs(hit) - 1);
  }
  // t = the lowest bf16 score of the list.  Certified: every admissible item outside the list has bf16 <= t,
  // hence fp32 <= t + eps < f_K; or the list is not full, i.e. it holds every admissible item.
  const float t = n_real > 0 ? p.cand_scores[static_cast<size_t>(b) * p.Kc + n_real - 1] : -INFINITY;
  const bool certified = n_real < p.Kc || f_k > __fadd_ru(t, eps);
  const int8_t path = bad ? 2 : (certified ? 0 : 1);
  if (path == 0) {
    const int k_eff = n_real < p.K ? n_real : p.K;
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      if (rank[q] < k_eff) {
        p.out_scores[static_cast<size_t>(b) * p.K + rank[q]] = s_sc[warp][lane + 32 * q];
        p.out_ids[static_cast<size_t>(b) * p.K + rank[q]] = s_id[warp][lane + 32 * q];
      }
    }
    if (lane == 0) p.out_cnt[b] = k_eff;
  }
  if (lane == 0) {
    p.path[b] = path;
    // every item of the fp32 top K (and every item tied with its K-th entry) has fp32 >= f_K, so bf16 >= f_K - eps
    p.tau[b] = path == 1 ? __fsub_rd(f_k, eps) : INFINITY;
    p.fk[b] = f_k;
  }
}

struct SelectParams {
  const int* users;          // [n] rows of the batch
  int n;
  const float* u;
  const float* table;
  const float* bias_pad;
  int rows, row_offset;
  const int* excl_sorted;    // [B][excl_stride] or null
  int excl_stride;
  const float* fk;           // [B] from lrb_exact_rescore
  int* cand_ids;             // [n][cap] collected ids (compacted in place)
  const int* cand_cnt;       // [n]
  int cap, K;
  float* out_scores;         // [B][K]
  int* out_ids;
  int* out_cnt;
  int8_t* path;
  float* ws_scores;          // [n][cap]
};

__global__ void __launch_bounds__(WARPS * 32) exact_select_kernel(const SelectParams p) {
  __shared__ float s_u[WARPS][D];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int i = blockIdx.x * WARPS + warp;
  if (i >= p.n) return;
  const int b = p.users[i];
  const int cnt = p.cand_cnt[i];
  if (cnt > p.cap) {                            // overflow: the fp32 path takes this user
    if (lane == 0) p.path[b] = 2;
    return;
  }
  s_u[warp][lane] = p.u[static_cast<size_t>(b) * D + lane];
  s_u[warp][lane + 32] = p.u[static_cast<size_t>(b) * D + lane + 32];
  __syncwarp();
  const float f_k = p.fk[b];
  const int* ex = p.excl_sorted ? p.excl_sorted + static_cast<size_t>(b) * p.excl_stride : nullptr;
  int* ids = p.cand_ids + static_cast<size_t>(i) * p.cap;
  float* scs = p.ws_scores + static_cast<size_t>(i) * p.cap;
  const unsigned lt_mask = (1u << lane) - 1u;

  // 1. drop history / out-of-shard ids, rescore, keep what can still rank (fp32 >= f_K <= the true K-th best)
  int ns = 0;
  bool bad = false;
  for (int base = 0; base < cnt; base += 32) {
    const int j = base + lane;
    const int id = j < cnt ? ids[j] : -1;
    const long long local = static_cast<long long>(id) - p.row_offset;
    bool ok = j < cnt && local >= 0 && local < p.rows;
    if (ok && ex != nullptr) {
      int lo = 0, hi = p.excl_stride;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(ex + mid) < id) lo = mid + 1; else hi = mid;
      }
      ok = !(lo < p.excl_stride && __ldg(ex + lo) == id);
    }
    const float s = ok ? score_f32(s_u[warp], p.table, p.bias_pad, static_cast<int>(local)) : -INFINITY;
    bad = bad || (ok && !finite(s));
    const bool keep = ok && s >= f_k;
    const unsigned bal = __ballot_sync(0xffffffffu, keep);
    __syncwarp();                               // (compaction writes only to positions <= those just read)
    if (keep) {
      const int idx = ns + __popc(bal & lt_mask);
      ids[idx] = id;
      scs[idx] = s;
    }
    ns += __popc(bal);
  }
  if (__any_sync(0xffffffffu, bad)) {
    if (lane == 0) p.path[b] = 2;
    return;
  }
  __syncwarp();

  // 2. K rounds of a warp-wide argmax by (score desc, id asc); collected ids are distinct
  int n_out = 0;
  for (int r = 0; r < p.K; ++r) {
    float bs = -INFINITY;
    int bi = INT_MAX, bj = -1;
    for (int j = lane; j < ns; j += 32) {
      const int id = ids[j];
      const float s = scs[j];
      if (id != INT_MAX && (bj < 0 || better(s, id, bs, bi))) { bs = s; bi = id; bj = j; }
    }
    float ws = bs;
    int wi = bi;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float os = __shfl_xor_sync(0xffffffffu, ws, o);
      const int oi = __shfl_xor_sync(0xffffffffu, wi, o);
      if (oi != INT_MAX && (wi == INT_MAX || better(os, oi, ws, wi))) { ws = os; wi = oi; }
    }
    if (wi == INT_MAX) break;
    if (lane == 0) {
      p.out_scores[static_cast<size_t>(b) * p.K + r] = ws;
      p.out_ids[static_cast<size_t>(b) * p.K + r] = wi;
    }
    if (bj >= 0 && bi == wi) ids[bj] = INT_MAX;
    __syncwarp();
    ++n_out;
  }
  if (lane == 0) p.out_cnt[b] = n_out;
}

}  // namespace exact
}  // namespace lrb

extern "C" {

int lrb_exact_rescore(const float* u, const float* table_f32, const float* bias_pad, const float* bound, int B,
                      int64_t rows, int64_t row_offset, const float* cand_scores, const int32_t* cand_ids, int Kc,
                      int K, float* out_scores, int32_t* out_ids, int32_t* out_cnt, int8_t* path, float* tau,
                      float* fk, void* stream) {
  using namespace lrb;
  int rc = check_arch();
  if (rc != LRB_OK) return rc;
  LRB_REQUIRE(u && table_f32 && bias_pad && bound && cand_scores && cand_ids && out_scores && out_ids && out_cnt &&
                  path && tau && fk, "lrb_exact_rescore: null pointer");
  LRB_REQUIRE(B > 0 && rows > 0 && row_offset >= 0 && rows + row_offset < INT_MAX, "lrb_exact_rescore: bad shape");
  LRB_REQUIRE(K >= 1 && K <= Kc && Kc <= LRB_MAX_K, "lrb_exact_rescore: need 1 <= K <= Kc <= %d", LRB_MAX_K);
  exact::RescoreParams p;
  p.u = u; p.table = table_f32; p.bias_pad = bias_pad; p.bound = bound;
  p.B = B; p.rows = static_cast<int>(rows); p.row_offset = static_cast<int>(row_offset);
  p.cand_scores = cand_scores; p.cand_ids = cand_ids; p.Kc = Kc; p.K = K;
  p.out_scores = out_scores; p.out_ids = out_ids; p.out_cnt = out_cnt; p.path = path; p.tau = tau; p.fk = fk;
  exact::exact_rescore_kernel<<<(B + exact::WARPS - 1) / exact::WARPS, exact::WARPS * 32, 0, as_stream(stream)>>>(p);
  LRB_CUDA_TRY(cudaGetLastError());
  return LRB_OK;
}

size_t lrb_exact_select_workspace_bytes(int n, int cap) {
  if (n < 1 || cap < 1) return 256;
  return (static_cast<size_t>(n) * cap * sizeof(float) + 255) & ~static_cast<size_t>(255);
}

int lrb_exact_select(const int32_t* users, int n, const float* u, const float* table_f32, const float* bias_pad,
                     int64_t rows, int64_t row_offset, const int32_t* excl_sorted, int excl_stride, const float* fk,
                     int32_t* cand_ids, const int32_t* cand_cnt, int cap, int K, float* out_scores,
                     int32_t* out_ids, int32_t* out_cnt, int8_t* path, void* workspace, size_t workspace_bytes,
                     void* stream) {
  using namespace lrb;
  int rc = check_arch();
  if (rc != LRB_OK) return rc;
  LRB_REQUIRE(users && u && table_f32 && bias_pad && fk && cand_cnt && out_scores && out_ids && out_cnt && path &&
                  workspace, "lrb_exact_select: null pointer");
  LRB_REQUIRE(cap >= 0 && (cap == 0 || cand_ids != nullptr), "lrb_exact_select: bad cap / cand_ids");
  LRB_REQUIRE(n > 0 && rows > 0 && row_offset >= 0 && rows + row_offset < INT_MAX, "lrb_exact_select: bad shape");
  LRB_REQUIRE(K >= 1 && K <= LRB_MAX_K, "lrb_exact_select: K must be in [1, %d]", LRB_MAX_K);
  LRB_REQUIRE(excl_sorted == nullptr || excl_stride > 0, "lrb_exact_select: bad excl_stride");
  const size_t need = lrb_exact_select_workspace_bytes(n, cap);
  if (workspace_bytes < need)
    return set_error(LRB_ERR_WORKSPACE, "lrb_exact_select: workspace %zu < %zu bytes", workspace_bytes, need);
  exact::SelectParams p;
  p.users = users; p.n = n; p.u = u; p.table = table_f32; p.bias_pad = bias_pad;
  p.rows = static_cast<int>(rows); p.row_offset = static_cast<int>(row_offset);
  p.excl_sorted = excl_sorted; p.excl_stride = excl_stride; p.fk = fk;
  p.cand_ids = cand_ids; p.cand_cnt = cand_cnt; p.cap = cap; p.K = K;
  p.out_scores = out_scores; p.out_ids = out_ids; p.out_cnt = out_cnt; p.path = path;
  p.ws_scores = static_cast<float*>(workspace);
  exact::exact_select_kernel<<<(n + exact::WARPS - 1) / exact::WARPS, exact::WARPS * 32, 0, as_stream(stream)>>>(p);
  LRB_CUDA_TRY(cudaGetLastError());
  return LRB_OK;
}

}  // extern "C"
