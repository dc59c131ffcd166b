// Train step of the retriever: loss value AND the gradient of every parameter, without the [B*L, N+1] logits tensor
// (SURVEY section 8f rank 2).
//
// Replaces LRUTrainer.calculate_loss + loss.backward():
//     logits = model(seqs).view(-1, N+1); loss = CrossEntropyLoss(ignore_index=0)(logits, labels.view(-1))
//                                                                 trainer/lru.py:20-28, trainer/base.py:107-111
// i.e. the backward of everything model/lru.py does:  embedding + LayerNorm (:57-60), per block the complex
// in_proj * gamma, the diagonal linear recurrence, Re(out_proj) + residual + LayerNorm (:149-161), the PFFN (:173-175),
// and the tied-embedding scoring matmul + bias (:85) under softmax cross-entropy.
//
// Dropout.  The four sites of model/lru.py (embedding :57-60, after out_proj :160, the PFFN hidden :174 and after
// w_2 :175) apply counter-based masks (common.cuh, DropoutSite): Philox4x32-10 of (seed, site, token, feature), so
// the backward recomputes them and oracle/dropout_oracle.py regenerates them.  torch's own dropout RNG stream is
// not reproduced.  Each mask is fused into a kernel that already touches the element: the gather / scatter of the
// embedding rows, the SGEMM epilogue before the residual add (backward: the LayerNorm backward writes the masked
// copy the GEMMs read), and the GELU forward / backward.  With every rate 0 nothing is evaluated or multiplied.
//
// Scope.  Training batches are LEFT-padded
// (dataloader/lru.py:98-118), for which the reference's recursive-doubling scan equals the recurrence
//     h_p = lambda * (mask_{p-1} h_{p-1}) + bu_p        (SURVEY probe P1),
// whose backward is the mirrored recurrence; a row with a zero after a non-zero id is rejected (error flag), and so
// is a label outside [0, rows) that is not ignore_index (torch's cross_entropy raises for one as well).
//
// fp32 throughout.  The gradients are compared with the reference's fp32 autograd at rtol 1e-3, and with the oracle
// run in float64 at 1e-4 of each tensor's largest entry (tests/test_gpu_train_encoder_paths.py).  Complex parameters are carried
// as (re, im) pairs, so the gradients that come out are (dL/dre, dL/dim) -- torch's convention for real-valued
// losses.  The softmax-CE backward recomputes the logits tile by tile in two passes (rows own dH, items own dE
// and dbias: no atomics on the big outputs, deterministic); everything between is small dense algebra over
// T = B*L tokens: one tiled SGEMM (NN / NT / TN) plus LayerNorm / GELU / gamma / scan kernels.
#include "api_util.h"
#include "common.cuh"

#include <climits>
#include <cmath>

namespace lrb {
namespace train {

constexpr int D = LRB_D;        // 64
constexpr int H2 = 2 * LRB_H;   // 256 reals = 128 complex channels, (re, im) interleaved
constexpr int FF = LRB_FF;      // 256
constexpr float LN_EPS = 1e-5f;
constexpr int ERR_NOT_LEFT_PADDED = 1;   // bits of the step's error flag
constexpr int ERR_BAD_LABEL = 2;

// packed weight / gradient blob (floats) -- the layout of llamarec_b200/packing.py and encode.cu
constexpr int OFF_EMB_LN_W = 0;
constexpr int OFF_EMB_LN_B = 64;
constexpr int OFF_BLOCKS = 128;
constexpr int B_LAM_RE = 0;
constexpr int B_LAM_IM = 128;
constexpr int B_GAMMA = 256;
constexpr int B_WIN_T = 384;                     // [64][256]
constexpr int B_BIN = B_WIN_T + D * H2;          // [256]
constexpr int B_WOUT_T = B_BIN + H2;             // [256][64]
constexpr int B_BOUT = B_WOUT_T + H2 * D;        // [64]
constexpr int B_LN1_W = B_BOUT + D;
constexpr int B_LN1_B = B_LN1_W + D;
constexpr int B_W1_T = B_LN1_B + D;              // [64][256]
constexpr int B_B1 = B_W1_T + D * FF;            // [256]
constexpr int B_W2_T = B_B1 + FF;                // [256][64]
constexpr int B_B2 = B_W2_T + FF * D;            // [64]
constexpr int B_LN2_W = B_B2 + D;
constexpr int B_LN2_B = B_LN2_W + D;
constexpr int BLOCK_FLOATS = B_LN2_B + D;

// ------------------------------------------------------------------------------------------------------------
// Tiled SGEMM, 64 x 64 output tile per CTA, 16 x 16 threads x (4 x 4) micro tile, K chunks of 16.
//   MODE 0 (NN): C[M][N]  = A[M][K] * W[K][N] (+ bias[N]) (+ R[M][N])          forward projections
//                with an active `drop`: C = mult (.) (A W + bias) + R   (dropout before the residual add)
//   MODE 1 (NT): C[M][K'] = A[M][N'] * W[K'][N']^T                              dX = dY * W^T   (here K' = rows of W)
//   MODE 2 (TN): C[K][N] += A[M][K]^T * G[M][N]  over an M slice (atomicAdd)    dW = X^T * dY
// ------------------------------------------------------------------------------------------------------------
constexpr int GT = 64;
constexpr int GK = 16;

template <int MODE>
__global__ void __launch_bounds__(256) sgemm_kernel(const float* __restrict__ A, const float* __restrict__ W,
                                                    const float* __restrict__ bias, const float* __restrict__ R,
                                                    float* __restrict__ C, int M, int N, int K, int m_per_cta,
                                                    DropoutSite drop) {
  __shared__ float sA[GK][GT + 1];
  __shared__ float sB[GK][GT + 1];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  if (MODE == 0 || MODE == 1) {
    // output C[M][NO], contraction length KC;  NN: NO = N, KC = K, B(k, n) = W[k][n];  NT: NO = K, KC = N, B(k, n) = W[n][k]
    const int NO = MODE == 0 ? N : K;
    const int KC = MODE == 0 ? K : N;
    const int m0 = blockIdx.y * GT, n0 = blockIdx.x * GT;
    for (int k0 = 0; k0 < KC; k0 += GK) {
      for (int e = threadIdx.x; e < GT * GK; e += 256) {
        const int r = e / GK, k = e % GK;          // A tile: rows m0.., columns k0..
        const int m = m0 + r;
        sA[k][r] = (m < M && k0 + k < KC) ? A[static_cast<size_t>(m) * KC + k0 + k] : 0.f;
      }
      for (int e = threadIdx.x; e < GT * GK; e += 256) {
        float v = 0.f;
        if (MODE == 0) {
          const int k = e / GT, n = e % GT;
          if (k0 + k < KC && n0 + n < NO) v = W[static_cast<size_t>(k0 + k) * N + n0 + n];
          sB[k][n] = v;
        } else {
          const int n = e / GK, k = e % GK;        // W[n0 + n][k0 + k], W is [K'][N'] = [NO][KC]
          if (k0 + k < KC && n0 + n < NO) v = W[static_cast<size_t>(n0 + n) * KC + k0 + k];
          sB[k][n] = v;
        }
      }
      __syncthreads();
#pragma unroll
      for (int k = 0; k < GK; ++k) {
        float a[4], b[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = sA[k][ty * 4 + i];
#pragma unroll
        for (int j = 0; j < 4; ++j) b[j] = sB[k][tx * 4 + j];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
      }
      __syncthreads();
    }
    const bool dropped = MODE == 0 && drop.active();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int m = m0 + ty * 4 + i;
      if (m >= M) continue;
      // the thread's four columns n0 + tx*4 .. +3 are one Philox group (n0 is a multiple of 64)
      float mult[4] = {1.f, 1.f, 1.f, 1.f};
      if (dropped) {
        const float4 d = dropout_mult4(drop, static_cast<uint32_t>(m), static_cast<uint32_t>((n0 + tx * 4) >> 2));
        mult[0] = d.x; mult[1] = d.y; mult[2] = d.z; mult[3] = d.w;
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int n = n0 + tx * 4 + j;
        if (n >= NO) continue;
        float v = acc[i][j];
        if (bias != nullptr) v += bias[n];
        if (dropped) v *= mult[j];
        if (R != nullptr) v += R[static_cast<size_t>(m) * NO + n];
        C[static_cast<size_t>(m) * NO + n] = v;
      }
    }
  } else {
    // TN: C[K][N] += sum over this CTA's slice of M of A[m][k] * G[m][n]   (A = X, W = dY)
    const int k0 = blockIdx.y * GT, n0 = blockIdx.x * GT;
    const int mb = blockIdx.z * m_per_cta;
    const int me = min(M, mb + m_per_cta);
    for (int m0 = mb; m0 < me; m0 += GK) {
      for (int e = threadIdx.x; e < GT * GK; e += 256) {
        const int mm = e / GT, c = e % GT;
        const int m = m0 + mm;
        sA[mm][c] = (m < me && k0 + c < K) ? A[static_cast<size_t>(m) * K + k0 + c] : 0.f;
        sB[mm][c] = (m < me && n0 + c < N) ? W[static_cast<size_t>(m) * N + n0 + c] : 0.f;
      }
      __syncthreads();
#pragma unroll
      for (int mm = 0; mm < GK; ++mm) {
        float a[4], b[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = sA[mm][ty * 4 + i];
#pragma unroll
        for (int j = 0; j < 4; ++j) b[j] = sB[mm][tx * 4 + j];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
      }
      __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int k = k0 + ty * 4 + i;
      if (k >= K) continue;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int n = n0 + tx * 4 + j;
        if (n < N) atomicAdd(C + static_cast<size_t>(k) * N + n, acc[i][j]);
      }
    }
  }
}

// column sums: db[n] += sum_m G[m][n]   (one CTA per 64-row slice, 256 threads walk the columns)
__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ G, float* __restrict__ db, int M, int N,
                                                      int m_per_cta) {
  const int mb = blockIdx.x * m_per_cta, me = min(M, mb + m_per_cta);
  for (int n = threadIdx.x; n < N; n += 256) {
    float s = 0.f;
    for (int m = mb; m < me; ++m) s += G[static_cast<size_t>(m) * N + n];
    atomicAdd(db + n, s);
  }
}

// ------------------------------------------------------------------------------------------------------------
// Embedding gather (+ monotone-mask check) and LayerNorm forward / backward over 64 features, one warp per row.
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gather_kernel(const void* __restrict__ ids, int id_bytes, int T, int L,
                                                     const float* __restrict__ table, long long table_rows,
                                                     float* __restrict__ out, unsigned char* __restrict__ mask,
                                                     int* __restrict__ err_flag, DropoutSite drop) {
  const int warp = (blockIdx.x * 256 + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= T) return;
  long long id = load_id(ids, warp, id_bytes);
  if (lane == 0) {
    mask[warp] = id > 0 ? 1 : 0;
    const int t = warp % L;
    // left padding only: a zero id must not follow a non-zero one inside a row
    if (t > 0 && id <= 0 && load_id(ids, warp - 1, id_bytes) > 0) atomicOr(err_flag, ERR_NOT_LEFT_PADDED);
  }
  if (id < 0 || id >= table_rows) id = 0;
  const float* row = table + static_cast<size_t>(id) * D;
  float v0 = row[lane], v1 = row[lane + 32];
  if (drop.active()) {   // embedding dropout: the stored row (the LayerNorm input) is mult (.) E[id]
    v0 *= dropout_mult(drop, warp, lane);
    v1 *= dropout_mult(drop, warp, lane + 32);
  }
  out[static_cast<size_t>(warp) * D + lane] = v0;
  out[static_cast<size_t>(warp) * D + lane + 32] = v1;
}

__global__ void __launch_bounds__(256) ln_fwd_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                     const float* __restrict__ b, float* __restrict__ y, int T) {
  const int warp = (blockIdx.x * 256 + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= T) return;
  const float v0 = x[static_cast<size_t>(warp) * D + lane], v1 = x[static_cast<size_t>(warp) * D + lane + 32];
  const float mean = warp_sum(v0 + v1) * (1.0f / 64.0f);
  const float d0 = v0 - mean, d1 = v1 - mean;
  const float var = warp_sum(d0 * d0 + d1 * d1) * (1.0f / 64.0f);
  const float rstd = 1.0f / sqrtf(var + LN_EPS);
  y[static_cast<size_t>(warp) * D + lane] = d0 * rstd * w[lane] + b[lane];
  y[static_cast<size_t>(warp) * D + lane + 32] = d1 * rstd * w[lane + 32] + b[lane + 32];
}

// dx = rstd * (g*w - mean(g*w) - xhat * mean(g*w*xhat));  dw += g * xhat;  db += g.   `x` is the LayerNorm INPUT.
// Each warp walks rows warp, warp + n_warps, ...; parameter gradients are reduced in registers, then one atomic each.
// If `dx_accum` the result is added to dx (a residual branch already left its gradient there).
// If `dx_drop` (only with an active `drop` and dx_accum == 0) it also receives mult (.) dx: the gradient that flows
// into the branch the dropout sits on, while dx itself is the residual branch's.
__global__ void __launch_bounds__(256) ln_bwd_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                     const float* __restrict__ g, float* __restrict__ dx,
                                                     float* __restrict__ dw, float* __restrict__ db, int T,
                                                     int dx_accum, float* __restrict__ dx_drop, DropoutSite drop) {
  const int n_warps = gridDim.x * 8;
  const int warp0 = (blockIdx.x * 256 + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  const float w0 = w[lane], w1 = w[lane + 32];
  float aw0 = 0.f, aw1 = 0.f, ab0 = 0.f, ab1 = 0.f;
  for (int r = warp0; r < T; r += n_warps) {
    const size_t o = static_cast<size_t>(r) * D;
    const float v0 = x[o + lane], v1 = x[o + lane + 32];
    const float mean = warp_sum(v0 + v1) * (1.0f / 64.0f);
    const float d0 = v0 - mean, d1 = v1 - mean;
    const float var = warp_sum(d0 * d0 + d1 * d1) * (1.0f / 64.0f);
    const float rstd = 1.0f / sqrtf(var + LN_EPS);
    const float h0 = d0 * rstd, h1 = d1 * rstd;
    const float g0 = g[o + lane], g1 = g[o + lane + 32];
    aw0 += g0 * h0; aw1 += g1 * h1; ab0 += g0; ab1 += g1;
    const float q0 = g0 * w0, q1 = g1 * w1;
    const float m1 = warp_sum(q0 + q1) * (1.0f / 64.0f);
    const float m2 = warp_sum(q0 * h0 + q1 * h1) * (1.0f / 64.0f);
    const float r0 = rstd * (q0 - m1 - h0 * m2), r1 = rstd * (q1 - m1 - h1 * m2);
    if (dx_accum) { dx[o + lane] += r0; dx[o + lane + 32] += r1; }
    else { dx[o + lane] = r0; dx[o + lane + 32] = r1; }
    if (dx_drop != nullptr) {
      dx_drop[o + lane] = r0 * dropout_mult(drop, r, lane);
      dx_drop[o + lane + 32] = r1 * dropout_mult(drop, r, lane + 32);
    }
  }
  atomicAdd(dw + lane, aw0); atomicAdd(dw + lane + 32, aw1);
  atomicAdd(db + lane, ab0); atomicAdd(db + lane + 32, ab1);
}

// scatter-add of the embedding-gather gradient: dTable[id] += mult (.) g[row]   (tied table: added to the scoring
// gradient; mult is the embedding-dropout multiplier, 1 without dropout)
__global__ void __launch_bounds__(256) scatter_rows_kernel(const void* __restrict__ ids, int id_bytes, int T,
                                                           long long table_rows, const float* __restrict__ g,
                                                           float* __restrict__ dtable, DropoutSite drop) {
  const int warp = (blockIdx.x * 256 + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= T) return;
  long long id = load_id(ids, warp, id_bytes);
  if (id < 0 || id >= table_rows) id = 0;
  float g0 = g[static_cast<size_t>(warp) * D + lane], g1 = g[static_cast<size_t>(warp) * D + lane + 32];
  if (drop.active()) {
    g0 *= dropout_mult(drop, warp, lane);
    g1 *= dropout_mult(drop, warp, lane + 32);
  }
  atomicAdd(dtable + static_cast<size_t>(id) * D + lane, g0);
  atomicAdd(dtable + static_cast<size_t>(id) * D + lane + 32, g1);
}

// ------------------------------------------------------------------------------------------------------------
// Elementwise: gamma scaling and exact-erf GELU
// ------------------------------------------------------------------------------------------------------------
// bu[t][2c + {0,1}] = pre[t][2c + {0,1}] * gamma[c]   (in place);  backward: dpre = dbu * gamma, dgamma[c] += sum dbu * pre
__global__ void __launch_bounds__(256) gamma_fwd_kernel(float* __restrict__ v, const float* __restrict__ gamma, long long n) {
  const long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x;
  if (i < n) v[i] *= gamma[(i & (H2 - 1)) >> 1];
}
// one CTA per slice of tokens, thread = real column (256): dgamma via bu = pre * gamma  =>  sum dbu * pre = sum dbu * bu / gamma
__global__ void __launch_bounds__(256) gamma_bwd_kernel(float* __restrict__ dbu, const float* __restrict__ bu,
                                                        const float* __restrict__ gamma, float* __restrict__ dgamma,
                                                        int T, int t_per_cta) {
  const int col = threadIdx.x;
  const float gm = gamma[col >> 1];
  const int tb = blockIdx.x * t_per_cta, te = min(T, tb + t_per_cta);
  float acc = 0.f;
  for (int t = tb; t < te; ++t) {
    const size_t o = static_cast<size_t>(t) * H2 + col;
    const float d = dbu[o];
    acc += d * bu[o];
    dbu[o] = d * gm;
  }
  atomicAdd(dgamma + (col >> 1), acc / gm);
}
// f, a, g are [T][FF]; one thread per four consecutive features (one Philox group of the hidden-dropout site)
LRB_DEVINL float gelu(float z) { return 0.5f * z * (1.0f + erff(z * 0.70710678118654752440f)); }
LRB_DEVINL float gelu_grad(float z) {   // d/dz [z Phi(z)] = Phi(z) + z phi(z)
  const float cdf = 0.5f * (1.0f + erff(z * 0.70710678118654752440f));
  const float pdf = 0.39894228040143267794f * expf(-0.5f * z * z);
  return cdf + z * pdf;
}
// a = mult (.) GELU(f)
__global__ void __launch_bounds__(256) gelu_fwd_kernel(const float4* __restrict__ f, float4* __restrict__ a, long long n4,
                                                       DropoutSite drop) {
  const long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x;
  if (i >= n4) return;
  const float4 z = f[i];
  float4 v = make_float4(gelu(z.x), gelu(z.y), gelu(z.z), gelu(z.w));
  if (drop.active()) {
    const float4 m = dropout_mult4(drop, static_cast<uint32_t>(i / (FF / 4)), static_cast<uint32_t>(i % (FF / 4)));
    v.x *= m.x; v.y *= m.y; v.z *= m.z; v.w *= m.w;
  }
  a[i] = v;
}
// da -> df in place:  df = mult (.) da (.) GELU'(f)
__global__ void __launch_bounds__(256) gelu_bwd_kernel(const float4* __restrict__ f, float4* __restrict__ g, long long n4,
                                                       DropoutSite drop) {
  const long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x;
  if (i >= n4) return;
  const float4 z = f[i];
  float4 d = g[i];
  if (drop.active()) {
    const float4 m = dropout_mult4(drop, static_cast<uint32_t>(i / (FF / 4)), static_cast<uint32_t>(i % (FF / 4)));
    d.x *= m.x; d.y *= m.y; d.z *= m.z; d.w *= m.w;
  }
  d.x *= gelu_grad(z.x); d.y *= gelu_grad(z.y); d.z *= gelu_grad(z.z); d.w *= gelu_grad(z.w);
  g[i] = d;
}
__global__ void __launch_bounds__(256) add_kernel(float* __restrict__ dst, const float* __restrict__ src, long long n) {
  const long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x;
  if (i < n) dst[i] += src[i];
}

// ------------------------------------------------------------------------------------------------------------
// The linear recurrence over time, one CTA (128 threads = complex channels) per user.
//   forward : h_p = lambda * (m_{p-1} h_{p-1}) + bu_p                 (h_0 = bu_0)
//   backward: G_p = g_p + conj(lambda) * m_p * G_{p+1}                (G_{L-1} = g_{L-1}),  dbu_p = G_p
//             dlambda += conj(m_{p-1} h_{p-1}) * G_p   written as real pairs:
//             h' = (lr a - li b, lr b + li a) with (a, b) = m h_{p-1}  =>  dlr += a Gr + b Gi,  dli += -b Gr + a Gi
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) scan_fwd_kernel(const float2* __restrict__ bu, float2* __restrict__ h,
                                                       const unsigned char* __restrict__ mask,
                                                       const float* __restrict__ lam_re, const float* __restrict__ lam_im,
                                                       int L) {
  const int b = blockIdx.x, c = threadIdx.x;
  const float lr = lam_re[c], li = lam_im[c];
  float pr = 0.f, pi = 0.f;   // m_{p-1} h_{p-1}
  for (int t = 0; t < L; ++t) {
    const size_t o = (static_cast<size_t>(b) * L + t) * LRB_H + c;
    const float2 u = bu[o];
    const float hr = pr * lr - pi * li + u.x;
    const float hi = pr * li + pi * lr + u.y;
    h[o] = make_float2(hr, hi);
    const float m = mask[b * L + t] ? 1.f : 0.f;
    pr = hr * m; pi = hi * m;
  }
}
// g (in): dL/dh, overwritten with dL/dbu
__global__ void __launch_bounds__(128) scan_bwd_kernel(float2* __restrict__ g, const float2* __restrict__ h,
                                                       const unsigned char* __restrict__ mask,
                                                       const float* __restrict__ lam_re, const float* __restrict__ lam_im,
                                                       float* __restrict__ dlam_re, float* __restrict__ dlam_im, int L) {
  const int b = blockIdx.x, c = threadIdx.x;
  const float lr = lam_re[c], li = lam_im[c];
  float Gr = 0.f, Gi = 0.f;     // G_{p+1}
  float dlr = 0.f, dli = 0.f;
  for (int t = L - 1; t >= 0; --t) {
    const size_t o = (static_cast<size_t>(b) * L + t) * LRB_H + c;
    const float m = mask[b * L + t] ? 1.f : 0.f;
    // G_p = g_p + m_p * conj(lambda) * G_{p+1}
    const float2 gp = g[o];
    const float cr = m * (lr * Gr + li * Gi), ci = m * (lr * Gi - li * Gr);
    Gr = gp.x + cr; Gi = gp.y + ci;
    g[o] = make_float2(Gr, Gi);
    if (t > 0) {
      const float mp = mask[b * L + t - 1] ? 1.f : 0.f;
      const float2 hp = h[o - LRB_H];
      const float a = mp * hp.x, bb = mp * hp.y;
      dlr += a * Gr + bb * Gi;
      dli += -bb * Gr + a * Gi;
    }
  }
  atomicAdd(dlam_re + c, dlr);
  atomicAdd(dlam_im + c, dli);
}
// (dL/dlam_re, dL/dlam_im, dL/dgamma) -> gradient of params_log = (nu_log, theta_log, gamma_log)   model/lru.py:151-152
//   lambda = exp(-exp(nu_log) + i exp(theta_log)),  gamma = exp(gamma_log)
__global__ void params_log_grad_kernel(float* __restrict__ gblk, const float* __restrict__ wblk,
                                       const float* __restrict__ params_log) {
  const int c = threadIdx.x;   // 128
  const float lr = wblk[B_LAM_RE + c], li = wblk[B_LAM_IM + c], gm = wblk[B_GAMMA + c];
  const float dlr = gblk[B_LAM_RE + c], dli = gblk[B_LAM_IM + c], dgm = gblk[B_GAMMA + c];
  const float nu = expf(params_log[c]);                  // exp(nu_log)
  const float theta = expf(params_log[LRB_H + c]);       // exp(theta_log)
  gblk[B_LAM_RE + c] = -(dlr * lr + dli * li) * nu;      // d nu_log
  gblk[B_LAM_IM + c] = (-dlr * li + dli * lr) * theta;   // d theta_log
  gblk[B_GAMMA + c] = dgm * gm;                          // d gamma_log
}

// ------------------------------------------------------------------------------------------------------------
// Softmax cross-entropy over the catalogue without the logits: forward statistics and the two backward passes.
// thread = hidden row (pass A) / item row (pass B) with its 64 values in registers, the other operand staged
// in shared memory 64 rows at a time.   g[m][n] = wgt_m * (exp(s_mn - lse_m) - [n == label_m])
// ------------------------------------------------------------------------------------------------------------
constexpr int CR = 128;   // rows (pass A) or items (pass B) per CTA
constexpr int CI = 64;    // staged rows of the other operand

// per row: lse over all items and the label's logit  ->  lse[m], row loss; loss_sum[0] += sum, loss_sum[1] += count.
// A label outside [0, rows) that is not ignore_index sets ERR_BAD_LABEL (the row is not counted by any pass).
__global__ void __launch_bounds__(CR) ce_stats_kernel(const float* __restrict__ hid, const float* __restrict__ table,
                                                      const float* __restrict__ bias, const long long* __restrict__ labels,
                                                      long long ignore_index, int M, int rows, float* __restrict__ lse,
                                                      float* __restrict__ loss_sum, int* __restrict__ err_flag) {
  __shared__ __align__(16) float sE[CI * D];
  __shared__ float sBias[CI];
  const int tid = threadIdx.x, m = blockIdx.x * CR + tid;
  const bool live = m < M;
  float u[D];
#pragma unroll
  for (int k = 0; k < D; ++k) u[k] = live ? hid[static_cast<size_t>(m) * D + k] : 0.f;
  const long long label = live ? labels[m] : -1;
  if (live && label != ignore_index && (label < 0 || label >= rows)) atomicOr(err_flag, ERR_BAD_LABEL);
  float run_max = -INFINITY, run_sum = 0.f, lab_logit = 0.f;
  for (int i0 = 0; i0 < rows; i0 += CI) {
    __syncthreads();
    for (int e = tid; e < CI * D; e += CR) sE[e] = (i0 + e / D < rows) ? table[static_cast<size_t>(i0) * D + e] : 0.f;
    if (tid < CI) sBias[tid] = i0 + tid < rows ? bias[i0 + tid] : -INFINITY;
    __syncthreads();
    const int nmax_i = min(CI, rows - i0);
    for (int j = 0; j < nmax_i; ++j) {
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
      for (int k = 0; k < D; k += 4) {
        a0 = fmaf(u[k], sE[j * D + k], a0); a1 = fmaf(u[k + 1], sE[j * D + k + 1], a1);
        a2 = fmaf(u[k + 2], sE[j * D + k + 2], a2); a3 = fmaf(u[k + 3], sE[j * D + k + 3], a3);
      }
      const float s = ((a0 + a1) + (a2 + a3)) + sBias[j];
      if (i0 + j == label) lab_logit = s;
      const float nm = fmaxf(run_max, s);
      run_sum = run_sum * expf(run_max - nm) + expf(s - nm);
      run_max = nm;
    }
  }
  float loss = 0.f, cnt = 0.f;
  if (live) {
    const float l = run_max + logf(run_sum);
    lse[m] = l;
    if (label != ignore_index && label >= 0 && label < rows) { loss = l - lab_logit; cnt = 1.f; }
  }
  loss = warp_sum(loss); cnt = warp_sum(cnt);
  if ((tid & 31) == 0 && cnt != 0.f) { atomicAdd(loss_sum, loss); atomicAdd(loss_sum + 1, cnt); }
}

// pass A: dH[m][:] = sum_n g[m][n] * E[n][:]     (grid: row tiles)
__global__ void __launch_bounds__(CR) ce_bwd_rows_kernel(const float* __restrict__ hid, const float* __restrict__ table,
                                                         const float* __restrict__ bias, const long long* __restrict__ labels,
                                                         long long ignore_index, const float* __restrict__ lse,
                                                         const float* __restrict__ loss_sum, int M, int rows,
                                                         float* __restrict__ dhid) {
  __shared__ __align__(16) float sE[CI * D];
  __shared__ float sBias[CI];
  const int tid = threadIdx.x, m = blockIdx.x * CR + tid;
  const bool live = m < M;
  float u[D], du[D];
#pragma unroll
  for (int k = 0; k < D; ++k) { u[k] = live ? hid[static_cast<size_t>(m) * D + k] : 0.f; du[k] = 0.f; }
  const long long label = live ? labels[m] : -1;
  const bool counted = live && label != ignore_index && label >= 0 && label < rows;
  const float wgt = counted ? 1.0f / loss_sum[1] : 0.f;    // mean over the counted rows
  const float l = live ? lse[m] : 0.f;
  for (int i0 = 0; i0 < rows; i0 += CI) {
    __syncthreads();
    for (int e = tid; e < CI * D; e += CR) sE[e] = (i0 + e / D < rows) ? table[static_cast<size_t>(i0) * D + e] : 0.f;
    if (tid < CI) sBias[tid] = i0 + tid < rows ? bias[i0 + tid] : -INFINITY;
    __syncthreads();
    if (!counted) continue;      // (after the barriers: every thread of the CTA takes part in the staging)
    const int nmax_i = min(CI, rows - i0);
    for (int j = 0; j < nmax_i; ++j) {
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
      for (int k = 0; k < D; k += 4) {
        a0 = fmaf(u[k], sE[j * D + k], a0); a1 = fmaf(u[k + 1], sE[j * D + k + 1], a1);
        a2 = fmaf(u[k + 2], sE[j * D + k + 2], a2); a3 = fmaf(u[k + 3], sE[j * D + k + 3], a3);
      }
      const float s = ((a0 + a1) + (a2 + a3)) + sBias[j];
      const float g = wgt * (expf(s - l) - (i0 + j == label ? 1.f : 0.f));
#pragma unroll
      for (int k = 0; k < D; ++k) du[k] = fmaf(g, sE[j * D + k], du[k]);
    }
  }
  if (live) {
#pragma unroll
    for (int k = 0; k < D; ++k) dhid[static_cast<size_t>(m) * D + k] = du[k];
  }
}

// pass B: dE[n][:] += sum_m g[m][n] * H[m][:],  dbias[n] += sum_m g[m][n]     (grid: item tiles x row slices)
__global__ void __launch_bounds__(CR) ce_bwd_items_kernel(const float* __restrict__ hid, const float* __restrict__ table,
                                                          const float* __restrict__ bias, const long long* __restrict__ labels,
                                                          long long ignore_index, const float* __restrict__ lse,
                                                          const float* __restrict__ loss_sum, int M, int rows,
                                                          int m_per_cta, float* __restrict__ dtable, float* __restrict__ dbias) {
  __shared__ __align__(16) float sH[CI * D];
  __shared__ float sLse[CI];
  __shared__ int sLab[CI];      // label if the row is counted, -1 otherwise
  const int tid = threadIdx.x, n = blockIdx.x * CR + tid;
  const bool live = n < rows;
  float e[D], de[D];
#pragma unroll
  for (int k = 0; k < D; ++k) { e[k] = live ? table[static_cast<size_t>(n) * D + k] : 0.f; de[k] = 0.f; }
  const float bn = live ? bias[n] : 0.f;
  const float inv_cnt = 1.0f / loss_sum[1];
  float db = 0.f;
  const int mb = blockIdx.y * m_per_cta, me = min(M, mb + m_per_cta);
  for (int m0 = mb; m0 < me; m0 += CI) {
    __syncthreads();
    for (int x = tid; x < CI * D; x += CR) sH[x] = (m0 + x / D < me) ? hid[static_cast<size_t>(m0) * D + x] : 0.f;
    if (tid < CI) {
      const int m = m0 + tid;
      long long lab = -1;
      if (m < me) { lab = labels[m]; if (lab == ignore_index || lab < 0 || lab >= rows) lab = -1; }
      sLab[tid] = static_cast<int>(lab);
      sLse[tid] = m < me ? lse[m] : 0.f;
    }
    __syncthreads();
    if (!live) continue;
    const int cnt = min(CI, me - m0);
    for (int j = 0; j < cnt; ++j) {
      const int lab = sLab[j];
      if (lab < 0) continue;     // ignored row: zero gradient (warp-uniform branch)
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
      for (int k = 0; k < D; k += 4) {
        a0 = fmaf(e[k], sH[j * D + k], a0); a1 = fmaf(e[k + 1], sH[j * D + k + 1], a1);
        a2 = fmaf(e[k + 2], sH[j * D + k + 2], a2); a3 = fmaf(e[k + 3], sH[j * D + k + 3], a3);
      }
      const float s = ((a0 + a1) + (a2 + a3)) + bn;
      const float g = inv_cnt * (expf(s - sLse[j]) - (lab == n ? 1.f : 0.f));
      db += g;
#pragma unroll
      for (int k = 0; k < D; ++k) de[k] = fmaf(g, sH[j * D + k], de[k]);
    }
  }
  if (live) {
#pragma unroll
    for (int k = 0; k < D; ++k) atomicAdd(dtable + static_cast<size_t>(n) * D + k, de[k]);
    atomicAdd(dbias + n, db);
  }
}

// keep[t][j] = 1 if element (t, j) of the site survives (the multiplier the kernels apply is non-zero)
__global__ void __launch_bounds__(256) dropout_mask_kernel(DropoutSite drop, int T, int width,
                                                           unsigned char* __restrict__ keep) {
  const int groups = (width + 3) / 4;
  const long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x;
  if (i >= static_cast<long long>(T) * groups) return;
  const int t = static_cast<int>(i / groups), j4 = static_cast<int>(i % groups);
  const float4 m = dropout_mult4(drop, static_cast<uint32_t>(t), static_cast<uint32_t>(j4));
  const float mv[4] = {m.x, m.y, m.z, m.w};
  for (int k = 0; k < 4 && 4 * j4 + k < width; ++k)
    keep[static_cast<size_t>(t) * width + 4 * j4 + k] = mv[k] != 0.f ? 1 : 0;
}

inline bool valid_rate(float p) { return p >= 0.f && p < 1.f; }   // false for NaN
inline DropoutSite make_site(uint64_t seed, int site, float p) {
  DropoutSite d;
  d.key0 = static_cast<uint32_t>(seed & 0xffffffffu);
  d.key1 = static_cast<uint32_t>(seed >> 32);
  d.site = static_cast<uint32_t>(site);
  d.thr = static_cast<uint32_t>(std::floor(static_cast<double>(p) * 4294967296.0));   // < 2^32 for p < 1
  d.scale = 1.0f / (1.0f - p);
  return d;
}

inline size_t al(size_t x) { return (x + 255) & ~static_cast<size_t>(255); }
inline unsigned blocks_for(long long n, int per) { return static_cast<unsigned>((n + per - 1) / per); }

}  // namespace train
}  // namespace lrb

extern "C" {

size_t lrb_train_workspace_bytes(int B, int L, int n_blocks) {
  using namespace lrb::train;
  if (B < 1 || L < 1 || n_blocks < 1) return 0;
  const size_t T = static_cast<size_t>(B) * L;
  // gathered rows + x0 ; per block: x_in is the previous output, bu, h, pre1, y, f1, a, pre2, out ; gradients: two
  // [T][64] ping-pong buffers and two [T][256] buffers ; lse ; mask ; error flag
  size_t per_block = 2 * al(T * H2 * 4) + 3 * al(T * D * 4) + 2 * al(T * FF * 4) + al(T * D * 4);
  return 2 * al(T * D * 4) + n_blocks * per_block + 3 * al(T * D * 4) + 2 * al(T * H2 * 4) + al(T * 4) + al(T) + 256;
}

int lrb_train_step(const void* ids, int id_bytes, const int64_t* labels, int B, int L, const float* table_f32,
                   int64_t table_rows, const float* bias_f32, const float* weights, const float* params_log,
                   int n_blocks, int64_t ignore_index,
                   float* loss_sum, float* grad_weights, float* grad_table, float* grad_bias, void* workspace,
                   size_t workspace_bytes, void* stream) {
  return lrb_train_step_dropout(ids, id_bytes, labels, B, L, table_f32, table_rows, bias_f32, weights, params_log,
                                n_blocks, ignore_index, loss_sum, grad_weights, grad_table, grad_bias, workspace,
                                workspace_bytes, stream, 0.f, 0.f, 0.f, 0);
}

int lrb_dropout_mask(uint64_t seed, int site, int T, int width, float p, uint8_t* keep, void* stream) {
  using namespace lrb;
  using namespace lrb::train;
  int rc = check_arch();
  if (rc != LRB_OK) return rc;
  LRB_REQUIRE(keep != nullptr, "lrb_dropout_mask: null pointer");
  LRB_REQUIRE(site >= 0 && T > 0 && width > 0, "lrb_dropout_mask: bad shape");
  LRB_REQUIRE(valid_rate(p), "lrb_dropout_mask: the rate must satisfy 0 <= p < 1");
  const long long n = static_cast<long long>(T) * ((width + 3) / 4);
  dropout_mask_kernel<<<blocks_for(n, 256), 256, 0, as_stream(stream)>>>(make_site(seed, site, p), T, width, keep);
  LRB_CUDA_TRY(cudaGetLastError());
  return LRB_OK;
}

int lrb_train_step_dropout(const void* ids, int id_bytes, const int64_t* labels, int B, int L, const float* table_f32,
                           int64_t table_rows, const float* bias_f32, const float* weights, const float* params_log,
                           int n_blocks, int64_t ignore_index,
                           float* loss_sum, float* grad_weights, float* grad_table, float* grad_bias, void* workspace,
                           size_t workspace_bytes, void* stream, float p_embed, float p_attn, float p_ffn,
                           uint64_t seed) {
  using namespace lrb;
  using namespace lrb::train;
  int rc = check_arch();
  if (rc != LRB_OK) return rc;
  LRB_REQUIRE(valid_rate(p_embed) && valid_rate(p_attn) && valid_rate(p_ffn),
              "lrb_train_step: dropout rates must satisfy 0 <= p < 1 (got %g, %g, %g)", p_embed, p_attn, p_ffn);
  LRB_REQUIRE(ids && labels && table_f32 && bias_f32 && weights && params_log && loss_sum && grad_weights &&
              grad_table && grad_bias && workspace, "lrb_train_step: null pointer");
  LRB_REQUIRE(B > 0 && L > 0 && n_blocks >= 1 && table_rows > 0 && table_rows < INT_MAX, "lrb_train_step: bad shape");
  LRB_REQUIRE(id_bytes == 4 || id_bytes == 8, "lrb_train_step: id_bytes must be 4 (int32) or 8 (int64)");
  if (L > LRB_MAX_LEN)
    return set_error(LRB_ERR_UNSUPPORTED, "sequence length %d exceeds LRB_MAX_LEN=%d", L, LRB_MAX_LEN);
  if (workspace_bytes < lrb_train_workspace_bytes(B, L, n_blocks))
    return set_error(LRB_ERR_WORKSPACE, "lrb_train_step: workspace too small");
  cudaStream_t st = as_stream(stream);
  const int T = B * L;
  const int rows = static_cast<int>(table_rows);
  const size_t n_w = static_cast<size_t>(OFF_BLOCKS) + static_cast<size_t>(n_blocks) * BLOCK_FLOATS;

  // ---- carve the workspace ----
  uint8_t* wsp = static_cast<uint8_t*>(workspace);
  auto take = [&](size_t bytes) { void* p = wsp; wsp += al(bytes); return p; };
  float* gath = static_cast<float*>(take(static_cast<size_t>(T) * D * 4));     // E[id]  (LayerNorm input)
  float* x0 = static_cast<float*>(take(static_cast<size_t>(T) * D * 4));
  struct Saved { float *bu, *h, *pre1, *y, *f1, *a, *pre2, *out; };
  Saved sv[8];
  LRB_REQUIRE(n_blocks <= 8, "lrb_train_step: at most 8 blocks");
  for (int i = 0; i < n_blocks; ++i) {
    sv[i].bu = static_cast<float*>(take(static_cast<size_t>(T) * H2 * 4));
    sv[i].h = static_cast<float*>(take(static_cast<size_t>(T) * H2 * 4));
    sv[i].pre1 = static_cast<float*>(take(static_cast<size_t>(T) * D * 4));
    sv[i].y = static_cast<float*>(take(static_cast<size_t>(T) * D * 4));
    sv[i].pre2 = static_cast<float*>(take(static_cast<size_t>(T) * D * 4));
    sv[i].f1 = static_cast<float*>(take(static_cast<size_t>(T) * FF * 4));
    sv[i].a = static_cast<float*>(take(static_cast<size_t>(T) * FF * 4));
    sv[i].out = static_cast<float*>(take(static_cast<size_t>(T) * D * 4));
  }
  float* g64a = static_cast<float*>(take(static_cast<size_t>(T) * D * 4));
  float* g64b = static_cast<float*>(take(static_cast<size_t>(T) * D * 4));
  float* g64c = static_cast<float*>(take(static_cast<size_t>(T) * D * 4));
  float* g256a = static_cast<float*>(take(static_cast<size_t>(T) * H2 * 4));
  float* g256b = static_cast<float*>(take(static_cast<size_t>(T) * H2 * 4));
  float* lse = static_cast<float*>(take(static_cast<size_t>(T) * 4));
  unsigned char* mask = static_cast<unsigned char*>(take(static_cast<size_t>(T)));
  int* err_flag = static_cast<int*>(take(16));

  // dropout sites (model/lru.py): 0 embedding (:57-60); per block i: 1+3i after out_proj (:160), 2+3i the PFFN
  // hidden (:174), 3+3i after w_2 (:175).  A site with p == 0 is inactive: no Philox, no multiply.
  const DropoutSite no_drop = make_site(0, 0, 0.f);
  const DropoutSite drop_embed = make_site(seed, 0, p_embed);
  auto drop_attn = [&](int i) { return make_site(seed, 1 + 3 * i, p_attn); };
  auto drop_hidden = [&](int i) { return make_site(seed, 2 + 3 * i, p_ffn); };
  auto drop_ffn_out = [&](int i) { return make_site(seed, 3 + 3 * i, p_ffn); };

  LRB_CUDA_TRY(cudaMemsetAsync(err_flag, 0, 4, st));
  LRB_CUDA_TRY(cudaMemsetAsync(loss_sum, 0, 2 * sizeof(float), st));
  LRB_CUDA_TRY(cudaMemsetAsync(grad_weights, 0, n_w * sizeof(float), st));
  LRB_CUDA_TRY(cudaMemsetAsync(grad_table, 0, static_cast<size_t>(rows) * D * sizeof(float), st));
  LRB_CUDA_TRY(cudaMemsetAsync(grad_bias, 0, static_cast<size_t>(rows) * sizeof(float), st));

  const unsigned warp_blocks = blocks_for(T, 8);          // one warp per row, 8 warps per CTA
  auto gemm_nn = [&](const float* A, const float* W, const float* bias, const float* R, float* C, int M, int N, int K,
                     const DropoutSite& drop) {
    dim3 grid(blocks_for(N, GT), blocks_for(M, GT));
    sgemm_kernel<0><<<grid, 256, 0, st>>>(A, W, bias, R, C, M, N, K, 0, drop);
  };
  auto gemm_nt = [&](const float* dY, const float* W, float* dX, int M, int N, int K) {   // dX[M][K] = dY[M][N] W[K][N]^T
    dim3 grid(blocks_for(K, GT), blocks_for(M, GT));
    sgemm_kernel<1><<<grid, 256, 0, st>>>(dY, W, nullptr, nullptr, dX, M, N, K, 0, no_drop);
  };
  const int m_slice = 1024;
  auto gemm_tn = [&](const float* X, const float* dY, float* dW, float* db, int M, int N, int K) {  // dW[K][N] += X^T dY
    dim3 grid(blocks_for(N, GT), blocks_for(K, GT), blocks_for(M, m_slice));
    sgemm_kernel<2><<<grid, 256, 0, st>>>(X, dY, nullptr, nullptr, dW, M, N, K, m_slice, no_drop);
    if (db != nullptr) colsum_kernel<<<blocks_for(M, m_slice), 256, 0, st>>>(dY, db, M, N, m_slice);
  };
  auto ew_blocks = [&](long long n) { return blocks_for(n, 256); };

  // =========================== forward (every intermediate the backward needs is kept) ===========================
  gather_kernel<<<warp_blocks, 256, 0, st>>>(ids, id_bytes, T, L, table_f32, table_rows, gath, mask, err_flag, drop_embed);
  ln_fwd_kernel<<<warp_blocks, 256, 0, st>>>(gath, weights + OFF_EMB_LN_W, weights + OFF_EMB_LN_B, x0, T);
  const float* x_in = x0;
  for (int i = 0; i < n_blocks; ++i) {
    const float* wb = weights + OFF_BLOCKS + static_cast<size_t>(i) * BLOCK_FLOATS;
    gemm_nn(x_in, wb + B_WIN_T, wb + B_BIN, nullptr, sv[i].bu, T, H2, D, no_drop);
    gamma_fwd_kernel<<<ew_blocks(static_cast<long long>(T) * H2), 256, 0, st>>>(sv[i].bu, wb + B_GAMMA, static_cast<long long>(T) * H2);
    scan_fwd_kernel<<<B, 128, 0, st>>>(reinterpret_cast<const float2*>(sv[i].bu), reinterpret_cast<float2*>(sv[i].h), mask,
                                       wb + B_LAM_RE, wb + B_LAM_IM, L);
    gemm_nn(sv[i].h, wb + B_WOUT_T, wb + B_BOUT, x_in, sv[i].pre1, T, D, H2, drop_attn(i));
    ln_fwd_kernel<<<warp_blocks, 256, 0, st>>>(sv[i].pre1, wb + B_LN1_W, wb + B_LN1_B, sv[i].y, T);
    gemm_nn(sv[i].y, wb + B_W1_T, wb + B_B1, nullptr, sv[i].f1, T, FF, D, no_drop);
    gelu_fwd_kernel<<<ew_blocks(static_cast<long long>(T) * FF / 4), 256, 0, st>>>(
        reinterpret_cast<const float4*>(sv[i].f1), reinterpret_cast<float4*>(sv[i].a), static_cast<long long>(T) * FF / 4,
        drop_hidden(i));
    gemm_nn(sv[i].a, wb + B_W2_T, wb + B_B2, sv[i].y, sv[i].pre2, T, D, FF, drop_ffn_out(i));
    ln_fwd_kernel<<<warp_blocks, 256, 0, st>>>(sv[i].pre2, wb + B_LN2_W, wb + B_LN2_B, sv[i].out, T);
    x_in = sv[i].out;
  }
  const float* hidden = x_in;
  const long long* lab = reinterpret_cast<const long long*>(labels);
  ce_stats_kernel<<<blocks_for(T, CR), CR, 0, st>>>(hidden, table_f32, bias_f32, lab, ignore_index, T, rows, lse, loss_sum,
                                                     err_flag);
  LRB_CUDA_TRY(cudaGetLastError());

  // =========================== backward ===========================
  float* dx = g64a;       // gradient w.r.t. the current block's output
  ce_bwd_rows_kernel<<<blocks_for(T, CR), CR, 0, st>>>(hidden, table_f32, bias_f32, lab, ignore_index, lse, loss_sum, T, rows, dx);
  {
    int sms = device_sm_count();
    if (sms <= 0) sms = 148;
    const unsigned item_tiles = blocks_for(rows, CR);
    unsigned slices = (2u * sms + item_tiles - 1) / item_tiles;
    const unsigned max_slices = blocks_for(T, 4 * CI);
    if (slices > max_slices) slices = max_slices;
    if (slices < 1) slices = 1;
    const int m_per = static_cast<int>((T + slices - 1) / slices);
    dim3 grid(item_tiles, blocks_for(T, m_per));
    ce_bwd_items_kernel<<<grid, CR, 0, st>>>(hidden, table_f32, bias_f32, lab, ignore_index, lse, loss_sum, T, rows, m_per,
                                             grad_table, grad_bias);
  }
  for (int i = n_blocks - 1; i >= 0; --i) {
    const float* wb = weights + OFF_BLOCKS + static_cast<size_t>(i) * BLOCK_FLOATS;
    float* gb = grad_weights + OFF_BLOCKS + static_cast<size_t>(i) * BLOCK_FLOATS;
    const float* xin = i == 0 ? x0 : sv[i - 1].out;
    float* dpre2 = g64b;
    float* dy = g64c;
    // out = LN2(pre2), pre2 = mult (.) (a W2 + b2) + y.  With dropout the W2 branch takes mult (.) dpre2, written
    // to g64c (free until dy is produced below); the residual branch takes dpre2 as it is.
    const DropoutSite d_out = drop_ffn_out(i);
    float* dpre2_w = d_out.active() ? g64c : dpre2;
    ln_bwd_kernel<<<148, 256, 0, st>>>(sv[i].pre2, wb + B_LN2_W, dx, dpre2, gb + B_LN2_W, gb + B_LN2_B, T, 0,
                                       d_out.active() ? dpre2_w : nullptr, d_out);
    gemm_tn(sv[i].a, dpre2_w, gb + B_W2_T, gb + B_B2, T, D, FF);
    gemm_nt(dpre2_w, wb + B_W2_T, g256a, T, D, FF);                     // da [T][256]
    gelu_bwd_kernel<<<ew_blocks(static_cast<long long>(T) * FF / 4), 256, 0, st>>>(
        reinterpret_cast<const float4*>(sv[i].f1), reinterpret_cast<float4*>(g256a), static_cast<long long>(T) * FF / 4,
        drop_hidden(i));                                                // -> df1
    gemm_tn(sv[i].y, g256a, gb + B_W1_T, gb + B_B1, T, FF, D);
    gemm_nt(g256a, wb + B_W1_T, dy, T, FF, D);                          // dy from the W1 branch
    add_kernel<<<ew_blocks(static_cast<long long>(T) * D), 256, 0, st>>>(dy, dpre2, static_cast<long long>(T) * D);   // + residual branch
    // y = LN1(pre1), pre1 = mult (.) (h W_out + b_out) + x_in.  The masked copy goes to g64a: dx was consumed by the
    // LN2 backward and is written again only by the in_proj branch below.
    float* dpre1 = g64b;
    const DropoutSite d_attn = drop_attn(i);
    float* dpre1_w = d_attn.active() ? g64a : dpre1;
    ln_bwd_kernel<<<148, 256, 0, st>>>(sv[i].pre1, wb + B_LN1_W, dy, dpre1, gb + B_LN1_W, gb + B_LN1_B, T, 0,
                                       d_attn.active() ? dpre1_w : nullptr, d_attn);
    gemm_tn(sv[i].h, dpre1_w, gb + B_WOUT_T, gb + B_BOUT, T, D, H2);
    gemm_nt(dpre1_w, wb + B_WOUT_T, g256b, T, D, H2);                   // dh [T][256]
    scan_bwd_kernel<<<B, 128, 0, st>>>(reinterpret_cast<float2*>(g256b), reinterpret_cast<const float2*>(sv[i].h), mask,
                                       wb + B_LAM_RE, wb + B_LAM_IM, gb + B_LAM_RE, gb + B_LAM_IM, L);        // -> dbu
    gamma_bwd_kernel<<<blocks_for(T, 256), 256, 0, st>>>(g256b, sv[i].bu, wb + B_GAMMA, gb + B_GAMMA, T, 256);   // -> d(pre-gamma)
    gemm_tn(xin, g256b, gb + B_WIN_T, gb + B_BIN, T, H2, D);
    gemm_nt(g256b, wb + B_WIN_T, dx, T, H2, D);                         // dx_in from the in_proj branch (dx is free now)
    add_kernel<<<ew_blocks(static_cast<long long>(T) * D), 256, 0, st>>>(dx, dpre1, static_cast<long long>(T) * D);   // + residual branch
    params_log_grad_kernel<<<1, 128, 0, st>>>(gb, wb, params_log + static_cast<size_t>(i) * 3 * LRB_H);
  }
  // x0 = LN_e(mult (.) E[id]): gath holds the dropped row, so the LayerNorm backward is unchanged
  ln_bwd_kernel<<<148, 256, 0, st>>>(gath, weights + OFF_EMB_LN_W, dx, g64b, grad_weights + OFF_EMB_LN_W,
                                     grad_weights + OFF_EMB_LN_B, T, 0, nullptr, no_drop);
  scatter_rows_kernel<<<warp_blocks, 256, 0, st>>>(ids, id_bytes, T, table_rows, g64b, grad_table, drop_embed);
  LRB_CUDA_TRY(cudaGetLastError());
  // input checks (one 4-byte read back: the step's result is meaningless otherwise)
  int err = 0;
  LRB_CUDA_TRY(cudaMemcpyAsync(&err, err_flag, 4, cudaMemcpyDeviceToHost, st));
  LRB_CUDA_TRY(cudaStreamSynchronize(st));
  if (err & ERR_BAD_LABEL)
    return set_error(LRB_ERR_BAD_ARG, "lrb_train_step: a label is outside [0, %d) and is not ignore_index %lld", rows,
                     static_cast<long long>(ignore_index));
  if (err & ERR_NOT_LEFT_PADDED)
    return set_error(LRB_ERR_UNSUPPORTED, "lrb_train_step: sequences must be left-padded (a zero id follows a non-zero id)");
  return LRB_OK;
}

}  // extern "C"
