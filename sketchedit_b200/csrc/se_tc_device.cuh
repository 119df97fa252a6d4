// Device-side building blocks shared by the tcgen05 convolution kernels (se_conv_tc.cu: NHWC input,
// se_conv_c8.cu: channel-blocked input): mbarrier / TMA / tcgen05 PTX wrappers and the fused epilogue.
#pragma once
#include <cuda_fp16.h>

#include "se_common.cuh"

namespace se {

// ------------------------------------------------------------------------------------------ PTX
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Bounded wait: a protocol bug traps after ~2 s of wall time (%globaltimer) instead of hanging the GPU box. The whole loop is
// ONE asm block on purpose: written as a C++ loop (per-lane `done` flag, early return, printf on timeout) ptxas treated
// everything after a wait as possibly divergent, kept every later value in vector registers and fed each tcgen05.mma operand
// through R2UR moves (4-7 per MMA; the stems' tensor pipe was 35 % active). (`tag` names the wait site; kept for debugging builds.)
#ifndef SE_WAIT_VARIANT
#define SE_WAIT_VARIANT 0
#endif
#if SE_WAIT_VARIANT == 1      // read the timer after every failed attempt
#define SE_WAIT_HINT ""
#define SE_WAIT_SPINS "1"
#elif SE_WAIT_VARIANT == 2    // let the hardware suspend the thread for up to ~2 us per attempt
#define SE_WAIT_HINT ", 2000"
#define SE_WAIT_SPINS "256"
#else
#define SE_WAIT_HINT ""
#define SE_WAIT_SPINS "256"
#endif
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, int tag) {
  (void)tag;
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 t0, t1;\n\t.reg .b32 n;\n\t"
      "mov.u64 t0, 0;\n\t"
      "OUTER_%=:\n\t"
      "mov.u32 n, 0;\n\t"
      "INNER_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1" SE_WAIT_HINT ";\n\t"
      "@p bra DONE_%=;\n\t"
      "add.u32 n, n, 1;\n\t"
      "setp.lt.u32 p, n, " SE_WAIT_SPINS ";\n\t"
      "@p bra INNER_%=;\n\t"
      "mov.u64 t1, %%globaltimer;\n\t"      // only after 256 failed attempts: the timer read is slow and must stay off the wake-up path
      "setp.eq.u64 p, t0, 0;\n\t"
      "@p mov.u64 t0, t1;\n\t"
      "sub.u64 t1, t1, t0;\n\t"
      "setp.lt.u64 p, t1, 2000000000;\n\t"
      "@p bra OUTER_%=;\n\t"
      "trap;\n\t"
      "DONE_%=:\n\t}"
      ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}

// same, acquiring at cluster scope: the barrier is signalled by threads of the peer CTA (CTA pairs)
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity, int tag) {
  (void)tag;
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 t0, t1;\n\t.reg .b32 n;\n\t"
      "mov.u64 t0, 0;\n\t"
      "OUTER_%=:\n\t"
      "mov.u32 n, 0;\n\t"
      "INNER_%=:\n\t"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1" SE_WAIT_HINT ";\n\t"
      "@p bra DONE_%=;\n\t"
      "add.u32 n, n, 1;\n\t"
      "setp.lt.u32 p, n, " SE_WAIT_SPINS ";\n\t"
      "@p bra INNER_%=;\n\t"
      "mov.u64 t1, %%globaltimer;\n\t"      // only after 256 failed attempts: the timer read is slow and must stay off the wake-up path
      "setp.eq.u64 p, t0, 0;\n\t"
      "@p mov.u64 t0, t1;\n\t"
      "sub.u64 t1, t1, t0;\n\t"
      "setp.lt.u64 p, t1, 2000000000;\n\t"
      "@p bra OUTER_%=;\n\t"
      "trap;\n\t"
      "DONE_%=:\n\t}"
      ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}

__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
// linear global -> shared bulk copy (bytes % 16 == 0), completion on an mbarrier
__device__ __forceinline__ void bulk_load_1d(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// warp index inside the CTA as a value the compiler KNOWS to be warp-uniform: built from vote results (a shuffle broadcast has
// the same value but is not recognised as uniform, so everything inside the role branches stayed on the vector datapath and
// every tcgen05.mma operand went through R2UR moves)
__device__ __forceinline__ int uniform_warp_index() {
  const int w = (int)(threadIdx.x >> 5);
  int r = 0;
#pragma unroll
  for (int k = 0; k < 5; ++k) r |= __any_sync(0xffffffffu, (w >> k) & 1) ? (1 << k) : 0;
  return r;
}

// one lane of a fully converged warp (the warp stays converged: the compiler keeps addresses / descriptors
// in uniform registers instead of broadcasting them lane by lane)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]^T, bf16 inputs, fp32 accumulate, M=128, N from idesc, K=16.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// predicated forms: the warp stays converged (no divergent branch around the issue sequence), so descriptor
// arithmetic stays on the uniform datapath; only the elected lane (lead != 0) actually issues
__device__ __forceinline__ void umma_bf16_if(uint32_t lead, uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.ne.b32 q, %5, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(lead)
      : "memory");
}
// same, descriptors passed as 32-bit halves (keeps the address arithmetic 32-bit / uniform)
__device__ __forceinline__ void umma_bf16_if32(uint32_t lead, uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                               uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t.reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "setp.ne.b32 q, %7, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}"
      ::"r"(tmem_d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate), "r"(lead)
      : "memory");
}
__device__ __forceinline__ void umma_commit_if(uint32_t lead, uint64_t* bar) {
  asm volatile(
      "{\n\t.reg .pred q;\n\t"
      "setp.ne.b32 q, %1, 0;\n\t"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}"
      ::"r"(smem_u32(bar)), "r"(lead)
      : "memory");
}

// ------------------------------------------------------------------------------------------ CTA pairs (cta_group::2)
// Two CTAs of a cluster (one TPC) execute ONE M=256 MMA: each supplies its own 128 rows of A and HALF of the B rows
// from its own shared memory (same offsets in both CTAs), accumulators land in each CTA's own TMEM. Only the
// leader (cluster rank 0) issues; TMA loads of both CTAs complete on the LEADER's mbarrier, commits are multicast.
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `bar` (a local shared::cta address) inside CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_rank(uint32_t local_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
  return r;
}
// RELAXED: every use signals "this accumulator stage has been drained" (tcgen05.wait::ld + tcgen05.fence::before_thread_sync precede it);
// nothing in generic memory is published by it. The default .release at cluster scope compiles to MEMBAR.ALL.GPU + ERRBAR, i.e. the
// epilogue warp sat until its output stores were visible GPU-wide before the MMA warp could get the TMEM stage back (ncu: 9 % of
// all warp samples of the CTA-pair kernels).
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// loads into OWN shared memory, completion bytes signalled on a (possibly remote) barrier of the CTA pair
__device__ __forceinline__ void tma_load_4d_pair(void* dst, const CUtensorMap* map, uint32_t bar_cluster_addr, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_pair(void* dst, const CUtensorMap* map, uint32_t bar_cluster_addr, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void umma2_bf16_if32(uint32_t lead, uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                                uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t.reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "setp.ne.b32 q, %7, 0;\n\t"
      "@q tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %5, p;\n\t}"
      ::"r"(tmem_d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate), "r"(lead)
      : "memory");
}
// arrives on the barrier at this offset in BOTH CTAs of the pair once the issued MMAs have completed
__device__ __forceinline__ void umma2_commit_if(uint32_t lead, uint64_t* bar) {
  asm volatile(
      "{\n\t.reg .pred q;\n\t.reg .b16 m;\n\t"
      "setp.ne.b32 q, %1, 0;\n\t"
      "mov.b16 m, 3;\n\t"
      "@q tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], m;\n\t}"
      ::"r"(smem_u32(bar)), "r"(lead)
      : "memory");
}

// mbarrier arrives once all previously issued MMAs of this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
// must be executed before the registers written by tmem_ld16 are read
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ float tanh_approx(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// write cnt (<= 16) consecutive channels of one pixel; static register indexing only (no local memory)
__device__ __forceinline__ void store_row_bf16(__nv_bfloat16* o, const float (&r)[16], int cnt, bool al8, bool al4) {
  if (cnt == 16 && al8) {
    *reinterpret_cast<uint4*>(o) = make_uint4(pack_bf16x2(r[0], r[1]), pack_bf16x2(r[2], r[3]), pack_bf16x2(r[4], r[5]), pack_bf16x2(r[6], r[7]));
    *reinterpret_cast<uint4*>(o + 8) = make_uint4(pack_bf16x2(r[8], r[9]), pack_bf16x2(r[10], r[11]), pack_bf16x2(r[12], r[13]), pack_bf16x2(r[14], r[15]));
  } else if (al4) {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (4 * j + 4 <= cnt) *reinterpret_cast<uint2*>(o + 4 * j) = make_uint2(pack_bf16x2(r[4 * j], r[4 * j + 1]), pack_bf16x2(r[4 * j + 2], r[4 * j + 3]));
#pragma unroll
    for (int i = 0; i < 16; ++i)
      if (i >= (cnt & ~3) && i < cnt) o[i] = __float2bfloat16(r[i]);
  } else {
#pragma unroll
    for (int i = 0; i < 16; ++i)
      if (i < cnt) o[i] = __float2bfloat16(r[i]);
  }
}
__device__ __forceinline__ void store_row_f32(float* o, const float (&r)[16], int cnt, bool al4) {
  if (cnt == 16 && al4) {
#pragma unroll
    for (int i = 0; i < 16; i += 4) *reinterpret_cast<float4*>(o + i) = make_float4(r[i], r[i + 1], r[i + 2], r[i + 3]);
  } else {
#pragma unroll
    for (int i = 0; i < 16; ++i)
      if (i < cnt) o[i] = r[i];
  }
}


#ifndef SE_EPI_GROUPS
#define SE_EPI_GROUPS 4
#endif
// Epilogue warps = 4 * groups (a group = 4 warps = the 128 TMEM lanes). The fused epilogue is latency bound (MUFU
// and TMEM-load dependency chains), so it wants warps, not ILP: with 2 groups (2 warps per scheduler) ncu shows the
// epilogue warps issuing on ~19 % of their cycles; 4 groups double the warps hiding each other's latencies. 640
// threads cap the kernel at 96 registers per thread.
constexpr int TC_EPI_GROUPS = SE_EPI_GROUPS;
constexpr int TC_NUM_THREADS = 128 + 128 * TC_EPI_GROUPS;   // 4 role warps + the epilogue groups (== TC_THREADS below)
constexpr int TC_TMEM_COLS = 512;
constexpr int TC_ACC_STRIDE = 256;   // TMEM columns between the two accumulator stages
constexpr int TC_MAX_STAGES = 8;

// ------------------------------------------------------------------------------------------ epilogue
// write up to 16 consecutive channels [c, c+cnt) of one output pixel; v[i >= cnt] must be 0 for C8 (pads are stored).
// kFast: the launch guarantees bf16 output and (C8, or NHWC with 16 B aligned rows and cnt in {8, 16}): the store is
// one or two 16 B vectors and nothing else (the epilogue runs one warp per scheduler: every instruction counts).
template <bool kFast>
__device__ __forceinline__ void epi_store16(const EpiParams& e, int img, int oy, int ox, int c, const float (&v)[16], int cnt) {
  if (e.out_c8) {
    // two channel blocks of 8: 16 B each, one plane (Hout*Wout*8 elements) apart
    __nv_bfloat16* base = reinterpret_cast<__nv_bfloat16*>(e.y);
    const size_t plane = (size_t)e.Hout * e.Wout * 8;
    const size_t o = (((size_t)img * e.ldo + ((e.choff + c) >> 3)) * e.Hout + oy) * e.Wout * 8 + (size_t)ox * 8;
    *reinterpret_cast<uint4*>(base + o) = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
    if (cnt > 8)
      *reinterpret_cast<uint4*>(base + o + plane) = make_uint4(pack_bf16x2(v[8], v[9]), pack_bf16x2(v[10], v[11]), pack_bf16x2(v[12], v[13]), pack_bf16x2(v[14], v[15]));
    return;
  }
  const size_t opix = ((size_t)img * e.Hout + oy) * e.Wout + ox;
  if (kFast) {
    __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(e.y) + opix * e.ldo + e.choff + c;
    *reinterpret_cast<uint4*>(o) = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
    if (cnt > 8)
      *reinterpret_cast<uint4*>(o + 8) = make_uint4(pack_bf16x2(v[8], v[9]), pack_bf16x2(v[10], v[11]), pack_bf16x2(v[12], v[13]), pack_bf16x2(v[14], v[15]));
    return;
  }
  const bool al4 = ((e.ldo | e.choff) & 3) == 0, al8 = ((e.ldo | e.choff) & 7) == 0;
  if (e.out_dt == DT_F32) store_row_f32(reinterpret_cast<float*>(e.y) + opix * e.ldo + e.choff + c, v, cnt, al4);
  else store_row_bf16(reinterpret_cast<__nv_bfloat16*>(e.y) + opix * e.ldo + e.choff + c, v, cnt, al8, al4);
}

// launch-time test for the minimal-instruction epilogue: bf16 output written as whole 16 B channel blocks
// (C8, or NHWC with 16 B aligned pixel rows and a channel count that is a multiple of 8)
__host__ __device__ inline bool epi_fast_ok(const EpiParams& e) {
  if (e.out_dt != DT_BF16) return false;
  if (e.out_c8) return true;
  const int n = (e.epi == EPI_LINEAR) ? e.Cout : (e.Cout >> 1);
  return ((e.ldo | e.choff) & 7) == 0 && (n % 8) == 0;
}

constexpr int TC_EPI_THREADS = 128 * TC_EPI_GROUPS;
constexpr int TC_THREADS = 128 + TC_EPI_THREADS;                   // warps 0-3: producer / MMA / TMEM alloc / 2nd MMA issuer

__device__ __forceinline__ float4 lds128(uint32_t saddr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr));
  return v;
}

// Epilogue constants in shared memory, three float arrays of `n` entries each, indexed by ACCUMULATOR COLUMN:
//   [0,n)  bias b    [n,2n)  b * log2(e) (ELU exponent)    [2n,3n)  0.5 * b (sigmoid-as-tanh argument)
// (gated layers: column c = feature c, column goff + c = its gate; see gated_column)
__device__ __forceinline__ void epi_fill_constants(float* cst, int n, const float* bias, const EpiParams& e, int tid, int nthreads) {
  const int half = e.Cout >> 1;
  for (int i = tid; i < n; i += nthreads) {
    int ch = i;   // output channel held by column i (-1: padding column)
    if (e.epi != EPI_LINEAR) ch = i < half ? i : (i >= e.goff && i < e.goff + half ? half + i - e.goff : -1);
    const float b = (bias != nullptr && ch >= 0 && ch < e.Cout) ? bias[ch] : 0.0f;
    cst[i] = b;
    cst[n + i] = b * 1.4426950408889634f;
    cst[2 * n + i] = 0.5f * b;
  }
}

// one gated output: act(f + b) * sigmoid(g + b')  (reference utils.py:29-32)
//   sigmoid(x) = 0.5 * tanh(0.5 x) + 0.5 (one MUFU); the accumulator column of a gate already holds 0.5 * g (the gate
//   weights are packed pre-multiplied by 0.5), hb = 0.5 * b'. ELU's exp as ex2: with the bias folded into the FMA (bl =
//   b * log2 e), or, kNoBl, as (f + b) * log2 e so that no third constant is needed (constant-bank epilogue).
template <bool kElu, bool kNoBl = false>
__device__ __forceinline__ float gate_one(float f, float ghalf, float b, float bl, float hb) {
  const float fv = f + b;
  float a;
  if (kElu) {
    const float ex = ex2_approx(kNoBl ? fv * 1.4426950408889634f : fmaf(f, 1.4426950408889634f, bl)) - 1.0f;
    a = fv > 0.0f ? fv : ex;
  } else {
    a = fmaxf(fv, 0.0f);
  }
  const float h = 0.5f * a;
  return fmaf(h, tanh_approx(ghalf + hb), h);
}

// Gated epilogue of one accumulator tile, minimal-instruction form (epi_fast_ok): work is cut in 8-column channel
// blocks (= one 16 B store); no masking is needed because padding columns hold zero weights and zero bias, so they
// come out as act(0) * sigmoid(0) = 0, which is exactly what the C8 padding channels must contain.
// nsplit == 1: this group drains the whole tile (16 columns at a time, 8 for an odd last block);
// nsplit  > 1: the tile has 3 * nsplit blocks, dealt to the groups 8 columns at a time.
template <bool kElu>
__device__ __forceinline__ void tc_epilogue_gated_fast(const EpiParams& e, const float* cst, int cst_n, uint32_t taddr, int img, bool valid,
                                                       int oy, int ox, int grp, int nsplit) {
  const int half = e.Cout >> 1, goff = e.goff;
  const int nb = (half + 7) >> 3;
  const uint32_t cs0 = smem_u32(cst);
  // all addressing in 32-bit units of 16 B (one 8-channel block of one pixel); the launchers check the tensor is < 2^32 units
  uint4* const ybase = reinterpret_cast<uint4*>(e.y);
  uint32_t obase, ostep;   // this pixel's first block / distance between consecutive blocks
  if (e.out_c8 == 2) {
    // space-to-depth for a stride-2 consumer: [N][4 * ldo/4 blocks][Hout/2][Wout/2][8], parity (oy&1, ox&1) selects
    // the block group, so the consumer's taps become plain stride-1 reads of one parity each
    const uint32_t Hs = e.Hout >> 1, Ws = e.Wout >> 1, par = ((oy & 1) << 1) | (ox & 1);
    ostep = Hs * Ws;
    obase = (((uint32_t)img * e.ldo + par * (uint32_t)e.par_stride + (e.choff >> 3)) * Hs + (oy >> 1)) * Ws + (ox >> 1);
  } else if (e.out_c8) {
    ostep = (uint32_t)e.Hout * e.Wout;
    obase = (((uint32_t)img * e.ldo + (e.choff >> 3)) * e.Hout + oy) * e.Wout + ox;
  } else {
    ostep = 1;
    obase = (((uint32_t)img * e.Hout + oy) * e.Wout + ox) * (e.ldo >> 3) + (e.choff >> 3);
  }
  // offset of output block b (fused layer pairs: the second layer's blocks sit blk_jump further on)
  auto boff = [&](int b) -> uint32_t { return obase + (uint32_t)b * ostep + (b >= e.blk_split ? (uint32_t)e.blk_jump : 0u); };
  // 4 outputs [c, c+4) from f[k..k+3], g[k..k+3]
  auto gate4 = [&](float* f, const float* g, int c, int k) {
    const float4 b = lds128(cs0 + c * 4), bl = lds128(cs0 + (cst_n + c) * 4), hb = lds128(cs0 + (2 * cst_n + goff + c) * 4);
    f[k] = gate_one<kElu>(f[k], g[k], b.x, bl.x, hb.x);
    f[k + 1] = gate_one<kElu>(f[k + 1], g[k + 1], b.y, bl.y, hb.y);
    f[k + 2] = gate_one<kElu>(f[k + 2], g[k + 2], b.z, bl.z, hb.z);
    f[k + 3] = gate_one<kElu>(f[k + 3], g[k + 3], b.w, bl.w, hb.w);
  };
  auto do16 = [&](int b) {
    const int c0 = b * 8;
    float f[16], g[16];
    tmem_ld16(taddr + c0, f);
    tmem_ld16(taddr + goff + c0, g);
    tmem_ld_wait();
    if (valid) {
#pragma unroll
      for (int q = 0; q < 4; ++q) gate4(f, g, c0 + 4 * q, 4 * q);
      ybase[boff(b)] = make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), pack_bf16x2(f[4], f[5]), pack_bf16x2(f[6], f[7]));
      ybase[boff(b + 1)] = make_uint4(pack_bf16x2(f[8], f[9]), pack_bf16x2(f[10], f[11]), pack_bf16x2(f[12], f[13]), pack_bf16x2(f[14], f[15]));
    }
  };
  auto do8 = [&](int b) {
    const int c0 = b * 8;
    float f[8], g[8];
    tmem_ld8(taddr + c0, f);
    tmem_ld8(taddr + goff + c0, g);
    tmem_ld_wait();
    if (valid) {
      gate4(f, g, c0, 0);
      gate4(f, g, c0 + 4, 4);
      ybase[boff(b)] = make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), pack_bf16x2(f[4], f[5]), pack_bf16x2(f[6], f[7]));
    }
  };
  if (nsplit == 1) {
    int b = 0;
    for (; b + 2 <= nb; b += 2) do16(b);
    if (b < nb) do8(b);
  } else {
    // three 8-column blocks per group (192-column tiles over 4 groups, nb == 3 * nsplit: c8_launch checks it): all six TMEM
    // loads are issued before the single wait, so their latency (long while the MMAs of the next tile stream accumulators)
    // is paid once, not 3x
    float f[3][8], g[3][8];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      tmem_ld8(taddr + (grp + j * nsplit) * 8, f[j]);
      tmem_ld8(taddr + goff + (grp + j * nsplit) * 8, g[j]);
    }
    tmem_ld_wait();
    if (valid) {
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        const int bb = grp + j * nsplit;
        gate4(f[j], g[j], bb * 8, 0);
        gate4(f[j], g[j], bb * 8 + 4, 4);
        ybase[boff(bb)] =
            make_uint4(pack_bf16x2(f[j][0], f[j][1]), pack_bf16x2(f[j][2], f[j][3]), pack_bf16x2(f[j][4], f[j][5]), pack_bf16x2(f[j][6], f[j][7]));
      }
    }
  }
}

// Split-half mode (DT_F16X2, the fp32-on-tensor-cores path): same gate, fp32-accurate math (ex2 / rcp approximations are good
// to ~2^-22; no tanh.approx), each output v stored as hi = fp16(64 v) and lo = fp16(64 v - hi), the lo block split_stride further on.
// The accumulator column of a gate still holds 0.5 * g (weights are packed pre-multiplied by 0.5, exact), hb = 0.5 * b'.
__device__ __forceinline__ float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// `s` = 1 / (activation scale * weight scale) of the split-half operands (se_common.cuh: kSplitActScale, ClassW::s_wscale).
// ELU's exp(x) - 1 cancels near 0 (ex2.approx is good to 2^-22 of exp(x), i.e. 2.4e-7 ABSOLUTE, 2.4e-4 of x = -1e-3):
// above -1/16 the degree-5 Taylor polynomial of expm1 is used instead (remainder < 1e-10).
template <bool kElu>
__device__ __forceinline__ float gate_one_exact(float f, float ghalf, float b, float hb, float s) {
  const float fv = fmaf(f, s, b);
  float a;
  if (kElu) {
    const float big = ex2_approx(fv * 1.4426950408889634f) - 1.0f;
    const float small = fv * fmaf(fv, fmaf(fv, fmaf(fv, fmaf(fv, 1.0f / 120.0f, 1.0f / 24.0f), 1.0f / 6.0f), 0.5f), 1.0f);
    a = fv > 0.0f ? fv : (fv > -0.0625f ? small : big);
  } else {
    a = fmaxf(fv, 0.0f);
  }
  const float gx = 2.0f * fmaf(ghalf, s, hb);
  return a * rcp_approx(1.0f + ex2_approx(-gx * 1.4426950408889634f));
}
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {
  __half2 v = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
template <bool kElu>
__device__ __forceinline__ void tc_epilogue_gated_split(const EpiParams& e, const float* cst, int cst_n, uint32_t taddr, int img, bool valid,
                                                        int oy, int ox, int grp, int nsplit) {
  const int half = e.Cout >> 1, goff = e.goff;
  const int nb = (half + 7) >> 3;
  uint4* const ybase = reinterpret_cast<uint4*>(e.y);
  uint32_t obase, ostep;
  if (e.out_c8 == 2) {
    const uint32_t Hs = e.Hout >> 1, Ws = e.Wout >> 1, par = ((oy & 1) << 1) | (ox & 1);
    ostep = Hs * Ws;
    obase = (((uint32_t)img * e.ldo + par * (uint32_t)e.par_stride + (e.choff >> 3)) * Hs + (oy >> 1)) * Ws + (ox >> 1);
  } else {
    ostep = (uint32_t)e.Hout * e.Wout;
    obase = (((uint32_t)img * e.ldo + (e.choff >> 3)) * e.Hout + oy) * e.Wout + ox;
  }
  for (int b = grp; b < nb; b += nsplit) {
    const int c0 = b * 8;
    float f[8], g[8];
    tmem_ld8(taddr + c0, f);
    tmem_ld8(taddr + goff + c0, g);
    tmem_ld_wait();
    if (valid) {
      uint32_t hi[4], lo[4];
#pragma unroll
      for (int k = 0; k < 8; k += 2) {
        float v0 = gate_one_exact<kElu>(f[k], g[k], cst[c0 + k], cst[2 * cst_n + goff + c0 + k], e.scale);
        float v1 = gate_one_exact<kElu>(f[k + 1], g[k + 1], cst[c0 + k + 1], cst[2 * cst_n + goff + c0 + k + 1], e.scale);
        v0 = fminf(fmaxf(v0 * kSplitActScale, -kSplitActMax), kSplitActMax);
        v1 = fminf(fmaxf(v1 * kSplitActScale, -kSplitActMax), kSplitActMax);
        const __half h0 = __float2half_rn(v0), h1 = __float2half_rn(v1);
        hi[k >> 1] = (uint32_t)__half_as_ushort(h0) | ((uint32_t)__half_as_ushort(h1) << 16);
        lo[k >> 1] = pack_f16x2(v0 - __half2float(h0), v1 - __half2float(h1));
      }
      const uint32_t o = obase + (uint32_t)b * ostep + (b >= e.blk_split ? (uint32_t)e.blk_jump : 0u);
      ybase[o] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
      ybase[o + (uint32_t)e.split_stride] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    }
  }
}

// Same epilogue for a whole tile of NB 8-column blocks with the constants in KERNEL PARAMETER space: NB is compile
// time, so every constant is an immediate constant-bank operand of its FMA/FADD and the epilogue issues no shared-memory
// loads (ncu: the first use of each LDS'd constant was the top stall of the small-N layers, short scoreboard).
// All TMEM loads of the tile are issued before the single wait.
template <bool kElu, int NB>
__device__ __forceinline__ void tc_epilogue_gated_const(const EpiParams& e, const float (&cst)[3][24], uint32_t taddr, int img, bool valid, int oy,
                                                        int ox, unsigned long long* trace = nullptr) {
  const int goff = e.goff;
  uint4* const ybase = reinterpret_cast<uint4*>(e.y);
  uint32_t obase, ostep;
  if (e.out_c8 == 2) {
    const uint32_t Hs = e.Hout >> 1, Ws = e.Wout >> 1, par = ((oy & 1) << 1) | (ox & 1);
    ostep = Hs * Ws;
    obase = (((uint32_t)img * e.ldo + par * (uint32_t)e.par_stride + (e.choff >> 3)) * Hs + (oy >> 1)) * Ws + (ox >> 1);
  } else if (e.out_c8) {
    ostep = (uint32_t)e.Hout * e.Wout;
    obase = (((uint32_t)img * e.ldo + (e.choff >> 3)) * e.Hout + oy) * e.Wout + ox;
  } else {
    ostep = 1;
    obase = (((uint32_t)img * e.Hout + oy) * e.Wout + ox) * (e.ldo >> 3) + (e.choff >> 3);
  }
  static_assert(NB <= 3, "one pass of at most three blocks (16 registers per block)");
  constexpr int PASS = NB;
#pragma unroll
  for (int b0 = 0; b0 < NB; b0 += PASS) {
    float f[PASS][8], g[PASS][8];
#pragma unroll
    for (int j = 0; j < PASS; ++j) {
      tmem_ld8(taddr + (b0 + j) * 8, f[j]);
      tmem_ld8(taddr + goff + (b0 + j) * 8, g[j]);
    }
    tmem_ld_wait();
    if (trace) *trace = clock64();
    if (valid) {
#pragma unroll
      for (int j = 0; j < PASS; ++j) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const int c = (b0 + j) * 8 + k;                // compile time
          f[j][k] = gate_one<kElu, true>(f[j][k], g[j][k], cst[0][c], 0.0f, cst[2][c]);   // both constants: immediate constant-bank operands
        }
        ybase[obase + (uint32_t)(b0 + j) * ostep] =
            make_uint4(pack_bf16x2(f[j][0], f[j][1]), pack_bf16x2(f[j][2], f[j][3]), pack_bf16x2(f[j][4], f[j][5]), pack_bf16x2(f[j][6], f[j][7]));
      }
    }
  }
}

// Drain one accumulator tile (this thread = TMEM lane = one output position) and apply the fused epilogue.
//   gated : out[c] = act(acc[c] + b[c]) * sigmoid(acc[goff + c] + b[Cout/2 + c])
//   linear: out[c] = (acc[c] + b[c]) * scale * colscale[img][c]
// The 16-column chunks of a tile are dealt round-robin to `nsplit` warp groups (this one is `grp`); nsplit == 1 means
// this group drains the whole tile (the groups then alternate tiles).
// (oy, ox): output pixel of this thread's position (the caller applies the output stride / sub-pixel offset).
template <bool kFast>
__device__ __forceinline__ void tc_epilogue_tile(const EpiParams& e, const float* cst, int cst_n, uint32_t taddr, int img, int nt, bool valid,
                                                 int oy, int ox, int grp, int nsplit = TC_EPI_GROUPS) {
  if (e.epi == EPI_LINEAR) {
    const int n0 = nt * e.NT;
    const float* cs = e.colscale ? e.colscale + (size_t)img * e.Cout : nullptr;
    for (int c0 = grp * 16; c0 < e.NT; c0 += 16 * nsplit) {
      const int cb = n0 + c0;
      if (cb >= e.Cout) break;
      float v[16];
      tmem_ld16(taddr + c0, v);
      tmem_ld_wait();
      if (valid) {
        const int cnt = min(16, e.Cout - cb);
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          float sc = e.scale;
          if (cs != nullptr && i < cnt) sc *= __ldg(cs + cb + i);
          v[i] = (i < cnt) ? (v[i] + (e.has_bias ? cst[cb + i] : 0.0f)) * sc : 0.0f;
        }
        epi_store16<kFast>(e, img, oy, ox, cb, v, cnt);
      }
    }
  } else if (kFast) {
    if (e.epi == EPI_GATE_ELU) tc_epilogue_gated_fast<true>(e, cst, cst_n, taddr, img, valid, oy, ox, grp, nsplit);
    else tc_epilogue_gated_fast<false>(e, cst, cst_n, taddr, img, valid, oy, ox, grp, nsplit);
  } else {
    // general form (fp32 or unaligned NHWC output: single-layer calls through the C ABI)
    const int half = e.Cout >> 1, goff = e.goff;
    const bool is_elu = (e.epi == EPI_GATE_ELU);
    for (int c0 = grp * 16; c0 < half; c0 += 16 * nsplit) {
      float f[16], g[16];
      tmem_ld16(taddr + c0, f);
      tmem_ld16(taddr + goff + c0, g);
      tmem_ld_wait();
      if (valid) {
        const int cnt = min(16, half - c0);
#pragma unroll
        for (int k = 0; k < 16; ++k) {
          const float b = cst[c0 + k], bl = cst[cst_n + c0 + k], hb = cst[2 * cst_n + goff + c0 + k];
          const float o = is_elu ? gate_one<true>(f[k], g[k], b, bl, hb) : gate_one<false>(f[k], g[k], b, bl, hb);
          f[k] = (k < cnt) ? o : 0.0f;
        }
        epi_store16<kFast>(e, img, oy, ox, c0, f, cnt);
      }
    }
  }
}

}  // namespace se
