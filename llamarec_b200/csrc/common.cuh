// Shared device-side helpers for the llamarec_b200 kernels (sm_100a only).
//
// Everything here is a thin wrapper over one PTX instruction (mbarrier, TMA,
// tcgen05, TMEM) or a small numeric helper shared by several kernels.  The
// bit layouts of the UMMA shared-memory / instruction descriptors follow the
// PTX ISA "tcgen05" chapter (the same layouts CUTLASS documents in
// cute/arch/mma_sm100_desc.hpp).
#pragma once

#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

#ifndef LRB_DEVINL
#define LRB_DEVINL __device__ __forceinline__
#endif

namespace lrb {

// ----------------------------------------------------------------------------
// Ordered-int encoding of floats (monotone: a < b  <=>  key(a) < key(b)).
// Used for atomicMax on score thresholds.
// ----------------------------------------------------------------------------
LRB_DEVINL int float_to_key(float f) {
  int i = __float_as_int(f);
  return i >= 0 ? i : (i ^ 0x7fffffff);
}
LRB_DEVINL float key_to_float(int k) {
  return __int_as_float(k >= 0 ? k : (k ^ 0x7fffffff));
}

// (score desc, id asc) ordering used everywhere a top-k list is built.
LRB_DEVINL bool better(float s_a, int id_a, float s_b, int id_b) {
  return (s_a > s_b) || (s_a == s_b && id_a < id_b);
}

LRB_DEVINL uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

LRB_DEVINL uint32_t elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(pred));
  return pred;
}

// ----------------------------------------------------------------------------
// mbarrier
// ----------------------------------------------------------------------------
LRB_DEVINL void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
LRB_DEVINL void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
LRB_DEVINL void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
LRB_DEVINL void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// The suspend-time hint lets the hardware park a waiting thread until the phase completes (or the hint expires)
// instead of returning after a few tens of cycles: a spinning try_wait + branch pair takes issue slots from the other
// warps of its SM sub-partition (scoring kernel, ncu round 2: 10 % of all issued instructions were such spins, and
// the epilogue warps that share a sub-partition with an MMA-issuing warp ran ~300 cycles per tile behind the others).
// (Same-box A/B on B200: the hint does not change the kernel's time either way; 20 us keeps a waiter parked for
// most of a hand-off and bounds what a missed wake-up could cost.)
#ifndef LRB_MBAR_SUSPEND_HINT
#define LRB_MBAR_SUSPEND_HINT 20000u
#endif
LRB_DEVINL bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2, %3;\n\t"
      "selp.b32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"(LRB_MBAR_SUSPEND_HINT)
      : "memory");
  return ok != 0;
}
LRB_DEVINL void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}

// ----------------------------------------------------------------------------
// TMA (cp.async.bulk[.tensor]) -- global -> shared, completion on an mbarrier
// ----------------------------------------------------------------------------
LRB_DEVINL void tma_prefetch_desc(const void* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
LRB_DEVINL void tma_load_2d(void* smem_dst, const void* tmap, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)),
      "r"(c0), "r"(c1)
      : "memory");
}
// 1-D bulk copy (no tensor map): bytes must be a multiple of 16, both sides 16-B aligned.
LRB_DEVINL void bulk_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes),
      "r"(smem_u32(bar))
      : "memory");
}

// ----------------------------------------------------------------------------
// tcgen05 / TMEM
// ----------------------------------------------------------------------------
LRB_DEVINL void tmem_alloc(uint32_t* smem_result, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_result)),
               "r"(ncols)
               : "memory");
}
LRB_DEVINL void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
LRB_DEVINL void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
LRB_DEVINL void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
LRB_DEVINL void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem] * B[smem], bf16 inputs, fp32 accumulate. One thread issues.
LRB_DEVINL void umma_bf16_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                             uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier once all previously issued tcgen05.mma of this thread retire.
LRB_DEVINL void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}
LRB_DEVINL void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Register budget of a warpgroup (4 consecutive warps; every warp of the group must execute the same instruction):
// the epilogue warpgroups of the scoring kernel take registers from the producer / MMA / service warpgroup.
template <int N>
LRB_DEVINL void setmaxnreg_inc() {
  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N));
}
template <int N>
LRB_DEVINL void setmaxnreg_dec() {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N));
}

// 32 lanes x 64 consecutive fp32 columns -> 64 registers per thread
LRB_DEVINL void tmem_ld_32x64(uint32_t taddr, uint32_t (&r)[64]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x64.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, "
      "%32, %33, %34, %35, %36, %37, %38, %39, %40, %41, %42, %43, %44, %45, %46, %47, "
      "%48, %49, %50, %51, %52, %53, %54, %55, %56, %57, %58, %59, %60, %61, %62, %63}, [%64];"
      :
        "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31]),
        "=r"(r[32]), "=r"(r[33]), "=r"(r[34]), "=r"(r[35]), "=r"(r[36]), "=r"(r[37]), "=r"(r[38]), "=r"(r[39]),
        "=r"(r[40]), "=r"(r[41]), "=r"(r[42]), "=r"(r[43]), "=r"(r[44]), "=r"(r[45]), "=r"(r[46]), "=r"(r[47]),
        "=r"(r[48]), "=r"(r[49]), "=r"(r[50]), "=r"(r[51]), "=r"(r[52]), "=r"(r[53]), "=r"(r[54]), "=r"(r[55]),
        "=r"(r[56]), "=r"(r[57]), "=r"(r[58]), "=r"(r[59]), "=r"(r[60]), "=r"(r[61]), "=r"(r[62]), "=r"(r[63])
      : "r"(taddr)
      : "memory");
}

// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread (thread i <-> TMEM lane base+i)
LRB_DEVINL void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
        "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}

// UMMA shared-memory matrix descriptor for a K-major bf16 tile whose rows are exactly one
// 128-byte swizzle atom wide (64 bf16): 8-row groups are 1024 B apart (SBO), LBO unused (=1),
// descriptor version 1 (sm_100), layout type 2 (SWIZZLE_128B).
LRB_DEVINL uint64_t umma_desc_k_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3ffff) >> 4);   // start address  [0,14)
  d |= static_cast<uint64_t>(1) << 16;                      // LBO (ignored)  [16,30)
  d |= static_cast<uint64_t>(1024 >> 4) << 32;              // SBO            [32,46)
  d |= static_cast<uint64_t>(1) << 46;                      // version        [46,48)
  d |= static_cast<uint64_t>(2) << 61;                      // SWIZZLE_128B   [61,64)
  return d;
}

// Instruction descriptor, kind::f16: D=f32, A=B=bf16, both K-major, shape M x N.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N) {
  return (1u << 4)                                  // c_format  = F32
         | (1u << 7)                                // a_format  = BF16
         | (1u << 10)                               // b_format  = BF16
         | (0u << 15) | (0u << 16)                  // a_major = b_major = K
         | (static_cast<uint32_t>(N >> 3) << 17)    // n_dim
         | (static_cast<uint32_t>(M >> 4) << 24);   // m_dim
}

// ----------------------------------------------------------------------------
// CTA pairs (cluster of 2, tcgen05 cta_group::2): one tcgen05.mma spans both SMs of a TPC.  Each CTA
// holds its own 128 accumulator rows and HALF of the B tile; the leader (cluster rank 0) issues the
// MMAs, its mbarriers collect the TMA bytes of both CTAs and the "accumulator drained" arrivals of
// both epilogues; tcgen05.commit multicasts "stage free" / "accumulator full" to both CTAs.
// ----------------------------------------------------------------------------
LRB_DEVINL uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
LRB_DEVINL void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `local` (a shared::cta address of this CTA) in CTA `rank` of the cluster
LRB_DEVINL uint32_t mapa_u32(uint32_t local, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local), "r"(rank));
  return r;
}
LRB_DEVINL void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
LRB_DEVINL void red_add_cluster_u32(uint32_t cluster_addr, uint32_t v) {
  asm volatile("red.relaxed.cluster.shared::cluster.add.u32 [%0], %1;" ::"r"(cluster_addr), "r"(v) : "memory");
}
// TMA load into THIS CTA's shared memory whose bytes are accounted on a barrier given as a
// shared::cluster address (the leader's barrier).
LRB_DEVINL void tma_load_2d_pair(void* smem_dst, const void* tmap, uint32_t bar_cluster_addr, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar_cluster_addr),
      "r"(c0), "r"(c1)
      : "memory");
}
// TMA load multicast to the CTAs of `cta_mask`: the tile lands at the same shared-memory offset in every destination
// CTA and its bytes are accounted on the mbarrier at the same offset of `bar` in every destination CTA.
LRB_DEVINL void tma_load_2d_mc(void* smem_dst, const void* tmap, uint64_t* bar, int c0, int c1, uint16_t cta_mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster"
      " [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)),
      "r"(c0), "r"(c1), "h"(cta_mask)
      : "memory");
}
// tcgen05.commit of a single-CTA MMA stream that arrives on the barrier at the same offset in every CTA of
// `cta_mask` (the shared-memory stage it frees is refilled by multicast loads of all of them).
LRB_DEVINL void umma_commit_mc(uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(smem_u32(bar)), "h"(cta_mask)
      : "memory");
}
LRB_DEVINL void tmem_alloc_pair(uint32_t* smem_result, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_result)),
               "r"(ncols)
               : "memory");
}
LRB_DEVINL void tmem_relinquish_pair() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
LRB_DEVINL void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
// D[tmem of both CTAs] (+)= A[smem, 128 rows per CTA] * B[smem, N/2 rows per CTA].  Leader thread only.
LRB_DEVINL void umma_bf16_ss_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                  uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on the barrier at the same shared-memory offset in every CTA of `cta_mask` once all
// previously issued tcgen05.mma of this thread retire.
LRB_DEVINL void umma_commit_pair(uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(smem_u32(bar)), "h"(cta_mask)
      : "memory");
}

// ----------------------------------------------------------------------------
// Packed fp32x2 add and 3-input max (both new on sm_100).
// ----------------------------------------------------------------------------
LRB_DEVINL void add_f32x2(float& a0, float& a1, float b0, float b1) {
  unsigned long long a, b, c;
  asm("mov.b64 %0, {%1, %2};" : "=l"(a) : "f"(a0), "f"(a1));
  asm("mov.b64 %0, {%1, %2};" : "=l"(b) : "f"(b0), "f"(b1));
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(c) : "l"(a), "l"(b));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a0), "=f"(a1) : "l"(c));
}
LRB_DEVINL float max3(float a, float b, float c) {
  float m;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(m) : "f"(a), "f"(b), "f"(c));
  return m;
}
LRB_DEVINL float min3(float a, float b, float c) {
  float m;
  asm("min.f32 %0, %1, %2, %3;" : "=f"(m) : "f"(a), "f"(b), "f"(c));
  return m;
}

// Log-depth reductions over small register arrays (3-input steps): the lock-step drain of the scoring kernel is a
// chain of dependent instructions executed by one or two warps per SM sub-partition, so depth, not count, is its cost.
template <int N>
LRB_DEVINL float tree_max(const float (&v)[N]) {
  if constexpr (N == 1) return v[0];
  else if constexpr (N == 2) return fmaxf(v[0], v[1]);
  else if constexpr (N == 3) return max3(v[0], v[1], v[2]);
  else {
    constexpr int M = (N + 2) / 3;
    float t[M];
#pragma unroll
    for (int i = 0; i < N / 3; ++i) t[i] = max3(v[3 * i], v[3 * i + 1], v[3 * i + 2]);
    if constexpr (N % 3 == 1) t[M - 1] = v[N - 1];
    if constexpr (N % 3 == 2) t[M - 1] = fmaxf(v[N - 2], v[N - 1]);
    return tree_max<M>(t);
  }
}
template <int N>
LRB_DEVINL float tree_min(const float (&v)[N]) {
  if constexpr (N == 1) return v[0];
  else if constexpr (N == 2) return fminf(v[0], v[1]);
  else if constexpr (N == 3) return min3(v[0], v[1], v[2]);
  else {
    constexpr int M = (N + 2) / 3;
    float t[M];
#pragma unroll
    for (int i = 0; i < N / 3; ++i) t[i] = min3(v[3 * i], v[3 * i + 1], v[3 * i + 2]);
    if constexpr (N % 3 == 1) t[M - 1] = v[N - 1];
    if constexpr (N % 3 == 2) t[M - 1] = fminf(v[N - 2], v[N - 1]);
    return tree_min<M>(t);
  }
}
template <int N>
LRB_DEVINL int tree_min_int(const int (&v)[N]) {
  if constexpr (N == 1) return v[0];
  else if constexpr (N == 2) return min(v[0], v[1]);
  else if constexpr (N == 3) return min(min(v[0], v[1]), v[2]);
  else {
    constexpr int M = (N + 2) / 3;
    int t[M];
#pragma unroll
    for (int i = 0; i < N / 3; ++i) t[i] = min(min(v[3 * i], v[3 * i + 1]), v[3 * i + 2]);
    if constexpr (N % 3 == 1) t[M - 1] = v[N - 1];
    if constexpr (N % 3 == 2) t[M - 1] = min(v[N - 2], v[N - 1]);
    return tree_min_int<M>(t);
  }
}
template <int N>
LRB_DEVINL int tree_sum_int(const int (&v)[N]) {
  if constexpr (N == 1) return v[0];
  else if constexpr (N == 2) return v[0] + v[1];
  else if constexpr (N == 3) return v[0] + v[1] + v[2];
  else {
    constexpr int M = (N + 2) / 3;
    int t[M];
#pragma unroll
    for (int i = 0; i < N / 3; ++i) t[i] = v[3 * i] + v[3 * i + 1] + v[3 * i + 2];
    if constexpr (N % 3 == 1) t[M - 1] = v[N - 1];
    if constexpr (N % 3 == 2) t[M - 1] = v[N - 2] + v[N - 1];
    return tree_sum_int<M>(t);
  }
}

// Explicit shared-space accessors (32-bit shared addresses).  The kernels carve dynamic shared
// memory from an integer-aligned base, which makes nvcc fall back to generic LD/ST otherwise.
LRB_DEVINL float4 lds_f32x4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "r"(addr)
               : "memory");
  return v;
}
LRB_DEVINL float lds_f32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
  return v;
}
LRB_DEVINL int lds_s32(uint32_t addr) {
  int v;
  asm volatile("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}
// re-read on every call (another warp may have raised the value), but a plain LDS -- not a generic LD
LRB_DEVINL int lds_volatile_s32(uint32_t addr) {
  int v;
  asm volatile("ld.volatile.shared.s32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}
LRB_DEVINL void sts_f32(uint32_t addr, float v) {
  asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
LRB_DEVINL void sts_s32(uint32_t addr, int v) {
  asm volatile("st.shared.s32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

// Item ids come as int64 (the reference's LongTensors) or int32 (DeviceEvalSet): `id_bytes` is 8 or 4.
LRB_DEVINL long long load_id(const void* __restrict__ ids, size_t idx, int id_bytes) {
  return id_bytes == 4 ? static_cast<long long>(__ldg(static_cast<const int*>(ids) + idx))
                       : __ldg(static_cast<const long long*>(ids) + idx);
}

LRB_DEVINL float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ----------------------------------------------------------------------------
// Counter-based dropout masks (train step).  Philox4x32-10 with the Random123 constants; the key is bumped
// between rounds.  Element (t, j) of site s -- t = b*L + l over the [B, L] batch, j the feature inside the
// site's width -- takes word (j & 3) of Philox(counter = (t, j >> 2, s, 0), key = (seed lo, seed hi)) and is
// kept iff that word >= thr = floor(p * 2^32); a kept element is multiplied by 1 / (1 - p) (fp32).  The masks
// are a pure function of (seed, s, t, j): the backward recomputes them, and oracle/dropout_oracle.py restates
// them bit for bit.
// ----------------------------------------------------------------------------
LRB_DEVINL uint4 philox4x32_10(uint4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r > 0) { k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
  }
  return c;
}

// One dropout site as the kernels see it.  thr == 0 (p == 0, or p below 2^-32) keeps every element with
// multiplier 1: kernels test `active()` and then evaluate no Philox and multiply by nothing.
struct DropoutSite {
  uint32_t key0, key1;   // seed & 0xffffffff, seed >> 32
  uint32_t site;
  uint32_t thr;          // floor(double(p) * 2^32)
  float scale;           // 1.0f / (1.0f - p)
  __host__ __device__ bool active() const { return thr != 0u; }
};

// multipliers of features 4*j4 .. 4*j4 + 3 of row t
LRB_DEVINL float4 dropout_mult4(const DropoutSite& d, uint32_t t, uint32_t j4) {
  const uint4 r = philox4x32_10(make_uint4(t, j4, d.site, 0u), d.key0, d.key1);
  return make_float4(r.x >= d.thr ? d.scale : 0.f, r.y >= d.thr ? d.scale : 0.f, r.z >= d.thr ? d.scale : 0.f,
                     r.w >= d.thr ? d.scale : 0.f);
}
// multiplier of feature j of row t
LRB_DEVINL float dropout_mult(const DropoutSite& d, uint32_t t, uint32_t j) {
  const float4 m = dropout_mult4(d, t, j >> 2);
  const uint32_t w = j & 3u;
  return w == 0 ? m.x : w == 1 ? m.y : w == 2 ? m.z : m.w;
}

}  // namespace lrb
