// tcgen05 implicit-GEMM convolution over CHANNEL-BLOCKED activations ("C8": [N][C/8][H][W][8] bf16) for sm_100a.
//
// Why this layout: 8 horizontally adjacent pixels of one channel block are 128 contiguous bytes = exactly one UMMA
// "core matrix" (8 rows x 16 B) of the no-swizzle K-major operand layout. So a spatial region of the input landed
// in shared memory by ONE TMA box [blocks][rows][cols*8] is directly usable as the A operand of EVERY tap of the
// convolution: the tap only changes the descriptor's start address (LBO = block plane size, SBO = row pitch).
//   * stride-1 convs with dilation <= 2 and the four sub-pixel classes of the x2 deconvs: the (16+2p) x (8+2p) halo
//     of a 16 x 8 output tile is loaded once per tile (double buffered) and re-used by all taps  ("HALO" mode;
//     A traffic drops from taps x tile to ~1.4 x tile, TMA row requests by >10x)
//   * dilation >= 4: one box per tap                                                           ("PERTAP" mode)
//   * 5x5 stems over the 8-channel packed input: GEMM-K runs over the pixel window (LBO = 16 B): 5 taps x 3 MMAs.
// The B operand (weights) is the pre-swizzled stage image of se_conv_tc.h, either streamed per k-step with
// cp.async.bulk or, when the whole layer fits (<= ~112 KB), loaded once and kept resident in shared memory.
//   * stride-2 3x3 layers read a SPACE-TO-DEPTH C8 tensor (written that way by the producer's epilogue): every tap is a
//     stride-1 read of one parity group, selected by a per-tap channel-block offset (C8Layer::tap_cb).
// Streamed-weight layers with N = 192 / 96 run as CTA PAIRS (cta_group::2, M = 256): each CTA loads half of every weight
// stage. 640 threads: warp 0 producer, warp 1 (+3 on resident layers) MMA issue, warp 2 TMEM allocation, warps 4-19 four
// epilogue groups; 2 / 4 / 8 TMEM accumulator stages for N <= 256 / 128 / 64. The fused epilogue lives in se_tc_device.cuh.
#include "se_conv_c8.h"

#include <stdlib.h>

#include <type_traits>
#include <vector>

#include "se_tc_device.cuh"

namespace se {

// SE_TC_DEBUG=2: per-tile timeline of CTA 0 (first 64 tiles of the non-fused resident path): dbg[2048 + iter * 8 + k] = clock64() at
//   k = 0 halo TMA issued, 1 issuer has the TMEM stage, 2 issuer has the halo (MMAs start), 3 MMAs + commits issued,
//   4 epilogue sees the accumulator, 5 TMEM drained + math + stores issued, 6 stage released
// Compiled in only with -DSE_C8_TRACE (SE_NVCC_EXTRA="-DSE_C8_TRACE" python -m sketchedit_b200.build --force): the extra live values cost
// the 96-register kernels 4-10 % on the small layers.
#ifdef SE_C8_TRACE
#define C8_TRACE(iter_, k_) do { if (p.dbg && p.trace && blockIdx.x == 0 && (iter_) < 64 && lane == 0) p.dbg[2048 + (iter_) * 8 + (k_)] = clock64(); } while (0)
#else
#define C8_TRACE(iter_, k_) do { } while (0)
#endif

constexpr int C8_TH = 16, C8_TW = 8;   // output tile: 16 rows x 8 columns = 128 positions

// no-swizzle K-major operand: core matrices of 8 rows x 16 B; LBO = next core matrix along K, SBO = along M
__device__ __forceinline__ uint64_t make_nosw_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;   // descriptor version 1 (sm_100); layout type 0 = no swizzle
  return d;
}
__device__ __forceinline__ uint64_t make_b_desc(uint32_t smem_addr, bool sw128) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)((sw128 ? 1024 : 512) >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)(sw128 ? 2 : 4) << 61;
  return d;
}

// R64 / R32 / MMAS: compile-time copies of p.r64 / p.r32 / p.mmas64 (R64 < 0: take them from p at run time).
// With compile-time trip counts the MMA issue sequence of a k-step is fully unrolled, so descriptor arithmetic of
// later MMAs overlaps the (long) issue latency of earlier ones: tools/bench/mma_rate.cu measures ~110 cycles per
// MMA for a rolled loop against the 40-96 cycle pipe time, i.e. a rolled loop starves the tensor core.
//
// PAIR = 1: the CTAs of a 2-CTA cluster work as one cta_group::2 unit on two tiles at a time (M = 256): every CTA
// loads the halo of ITS tile but only HALF of each weight stage (rows [rank*NT/2, +NT/2) through the 2-D tensor map
// tmB over the pair-format image), which halves the streamed-weight ingest that bounds the 96->192 layers, and the
// leader issues one MMA for both tiles. Streaming (non-resident) layers only.
//
// KS1 = 1: the layer has ONE k-step per tile (resident weights + halo: r64/r32 are all its K units). Everything that
// depends on the k-step index (A-offset table index, accumulate flag, last-step test, resident B address) is then a
// compile-time constant, so the issue sequence is just "constant-bank offset + base -> descriptor -> MMA": the
// indexed constant loads of the generic form (~100+ cycles each, on the critical path of a 15-18 MMA tile) disappear.
//
// NCLS > 1 (2 or 4; KS1 layers only): fused sub-pixel classes of a x2 deconv (C8Group). The persistent loop runs over
// VIRTUAL tiles v = tile * NCLS + class: the producer loads one (union) halo per real tile; the two MMA issuers take
// alternate virtual tiles (issuer `me` gets the classes of its parity) and each commits the halo buffer back after its last
// class of the tile (a_empty counts 2 arrivals); TMEM stages and epilogue groups are indexed by v, so with NCLS = 4 epilogue
// group g always drains class g. A class selects its resident weight image (cls_bytes apart), its A-offset row
// aoff[class * C8_CLS_UNITS + unit] (compile-time class index -> constant-bank operands) and its output sub-pixel offset.
template <int R64, int R32, int MMAS, int PAIR, int KS1 = 0, int NCLS = 1>
__global__ void __launch_bounds__(TC_NUM_THREADS, 1)
conv_c8_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const C8Params p) {
  constexpr bool kPair = PAIR != 0;
  const uint32_t cta_rank = kPair ? cluster_ctarank() : 0u;
  const int r64 = R64 >= 0 ? R64 : p.r64, r32 = R64 >= 0 ? R32 : p.r32, mmas64 = R64 >= 0 ? MMAS : p.mmas64;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  // carve: [halo A buffers][resident weights][stages: (tap A box) + (B image)] [barriers][tmem ptr][bias]
  const bool halo = (p.mode == C8_HALO);
  const int NTl = kPair ? p.NT / 2 : p.NT;                   // B rows held by this CTA
  const int b64_bytes = NTl * 128, b32_bytes = NTl * 64;
  const int b_bytes = r64 * b64_bytes + r32 * b32_bytes;
  const int stage_a = halo ? 0 : p.a_bytes;
  const int stage_b = p.resident ? 0 : b_bytes;
  const int stage_bytes = stage_a + stage_b;
  uint8_t* sHalo = smem;
  uint8_t* sWres = sHalo + (halo ? p.a_bufs * p.a_bytes : 0);
  uint8_t* sStages = sWres + (p.resident ? p.wres_bytes : 0);
  uint8_t* tail = sStages + (size_t)p.num_stages * stage_bytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(tail);
  uint64_t* empty_bar = full_bar + TC_MAX_STAGES;
  uint64_t* a_full = empty_bar + TC_MAX_STAGES;
  uint64_t* a_empty = a_full + C8_MAX_ABUFS;
  uint64_t* tmem_full = a_empty + C8_MAX_ABUFS;
  uint64_t* tmem_empty = tmem_full + 8;
  uint64_t* wres_bar = tmem_empty + 8;
  // accumulator ring: N <= 128 leaves room for 4 TMEM stages: the four epilogue groups drain alternate tiles (a group
  // has four tile-times per tile); wider tiles keep 2 stages and split a tile's columns between the groups.
  // N <= 64 even fits 8 stages, two per group: while a group drains tile i the MMAs of tile i+4 already fill its second
  // stage, so a group's cycle is the drain alone instead of drain + MMA latency (the small-N layers are epilogue bound)
  // (the launcher picks the ring sizes, all powers of two - see c8_launch)
  const int acc_stages = p.acc_stages, acc_stride = p.acc_stride;
  const int epi_split = p.epi_split;
  // slot / phase parity of iteration i in a ring of n = 2^shift slots
  auto ring_of = [](int i, int n, int shift, int& slot, uint32_t& phase) {
    slot = i & (n - 1);
    phase = (uint32_t)(i >> shift) & 1u;
  };
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(wres_bar + 1);
  float* bias_s = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(tmem_ptr_smem + 4) + 15) & ~uintptr_t(15));   // 16 B aligned: read with ld.shared.v4

  // warp-uniform by construction (a shuffle from lane 0): lets the compiler keep role-dependent values - the tile
  // parity of the second MMA issuer, ring indices, descriptors - on the uniform datapath
  const int warp = uniform_warp_index();
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA)) : "memory");
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < TC_MAX_STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < C8_MAX_ABUFS; ++i) {
      mbar_init(&a_full[i], 1);
      mbar_init(&a_empty[i], NCLS > 1 ? 2 : 1);   // fused classes: one commit per MMA issuer
    }
    for (int i = 0; i < 8; ++i) {
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], (kPair ? 2 : 1) * 4 * epi_split);   // one arrive per epilogue warp (pair: of both CTAs)
    }
    mbar_init(wres_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    if (kPair) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)), "r"(TC_TMEM_COLS) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)), "r"(TC_TMEM_COLS) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  const int cst_n = p.NT + 32;
  epi_fill_constants(bias_s, cst_n, p.bias, p.e, threadIdx.x, TC_NUM_THREADS);
  tc_fence_before();
  if (kPair) cluster_sync_all(); else __syncthreads();       // pair: the peer's barriers must exist before any remote signal
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_ptr_smem, 0);   // uniform copy (feeds MMA / tcgen05.ld addresses)

  const int total_tiles = p.N * p.tiles_x * p.tiles_y;
  const int ksteps = p.ksteps;
  const bool staged = stage_bytes > 0;

  if (warp == 0) {
    // ==================================================================== producer
    if (p.resident && elect_one()) {
      // whole layer's weights, once: bulk copies of <= 64 KB
      mbar_expect_tx(wres_bar, (uint32_t)p.wres_bytes);
      for (int off = 0; off < p.wres_bytes; off += 65536) {
        const int n = min(65536, p.wres_bytes - off);
        bulk_load_1d(sWres + off, p.w + off, (uint32_t)n, wres_bar);
      }
    }
    __syncwarp();
    int stage = 0, iter = 0;
    uint32_t phase = 0;
    long long t_wait = 0, t_begin = clock64();
    // tile coordinates advance incrementally by gridDim.x tiles (mixed radix step), no per-tile integer division
    int tx = blockIdx.x % p.tiles_x, ty = (blockIdx.x / p.tiles_x) % p.tiles_y, img = blockIdx.x / (p.tiles_x * p.tiles_y);
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++iter) {
      if (tile != (int)blockIdx.x) {
        tx += p.step_x;
        if (tx >= p.tiles_x) { tx -= p.tiles_x; ++ty; }
        ty += p.step_y;
        if (ty >= p.tiles_y) { ty -= p.tiles_y; ++img; }
        img += p.step_img;
      }
      const int x0 = tx * C8_TW, y0 = ty * C8_TH;
      if (halo) {
        int ab;
        uint32_t aphase;
        ring_of(iter, p.a_bufs, p.a_shift, ab, aphase);
        const long long tw = p.dbg ? clock64() : 0;
        mbar_wait(&a_empty[ab], aphase ^ 1, 5);
        if (p.dbg) t_wait += clock64() - tw;
        if (elect_one()) {
          if (kPair) {
            if (cta_rank == 0) mbar_expect_tx(&a_full[ab], 2u * (uint32_t)p.a_tx_bytes);
            tma_load_4d_pair(sHalo + (size_t)ab * p.a_bytes, &tmA, mapa_rank(smem_u32(&a_full[ab]), 0), (x0 - p.pad_x0) * 8, y0 - p.pad_y0,
                             p.x_cb_off, img);
          } else {
            mbar_expect_tx(&a_full[ab], (uint32_t)p.a_tx_bytes);
            tma_load_4d(sHalo + (size_t)ab * p.a_bytes, &tmA, &a_full[ab], (x0 - p.pad_x0) * 8, y0 - p.pad_y0, p.x_cb_off, img);
          }
        }
        __syncwarp();
        C8_TRACE(iter, 0);
      }
      if (staged) {
        for (int ks = 0; ks < ksteps; ++ks) {
          const long long tw = p.dbg ? clock64() : 0;
          mbar_wait(&empty_bar[stage], phase ^ 1, 1);
          if (p.dbg) t_wait += clock64() - tw;
          uint8_t* st = sStages + (size_t)stage * stage_bytes;
          if (elect_one()) {
            if (kPair) {
              const uint32_t lead_bar = mapa_rank(smem_u32(&full_bar[stage]), 0);
              if (cta_rank == 0) mbar_expect_tx(&full_bar[stage], 2u * (uint32_t)((halo ? 0 : p.a_tx_bytes) + stage_b));
              tma_load_2d_pair(st + stage_a, &tmB, lead_bar, 0, (ks * 2 + (int)cta_rank) * (b_bytes >> 9));   // 512 B rows
              if (!halo) tma_load_4d_pair(st, &tmA, lead_bar, (x0 + p.dx[ks]) * 8, y0 + p.dy[ks], p.x_cb_off + p.tap_cb[ks], img);
            } else {
              mbar_expect_tx(&full_bar[stage], (uint32_t)((halo ? 0 : p.a_tx_bytes) + stage_b));
              if (!p.resident) bulk_load_1d(st + stage_a, p.w + (size_t)ks * b_bytes, (uint32_t)b_bytes, &full_bar[stage]);
              if (!halo) {   // PERTAP: a stage is exactly one tap
                tma_load_4d(st, &tmA, &full_bar[stage], (x0 + p.dx[ks]) * 8, y0 + p.dy[ks], p.x_cb_off + p.tap_cb[ks], img);
              }
            }
          }
          __syncwarp();
          if (++stage == p.num_stages) { stage = 0; phase ^= 1; }
        }
      }
    }
    if (p.dbg && lane == 0) { p.dbg[blockIdx.x * 8 + 0] = t_wait; p.dbg[blockIdx.x * 8 + 1] = clock64() - t_begin; }
  } else if ((warp == 1 || (warp == 3 && !staged)) && (!kPair || cta_rank == 0)) {
    // ==================================================================== MMA issuer (pair: the leader, for both CTAs)
    // Nothing streamed per k-step (resident weights + halo): a tile is ONE short burst of MMAs, and the issuer's
    // per-tile protocol (two commits, two barrier waits, fence, descriptor set-up: ~600 cycles measured) is longer
    // than the 3-4 queued MMAs of a small-N layer (40-56 cycles each) can cover, so the tensor pipe would idle
    // between tiles. Warps 1 and 3 therefore issue alternate tiles: each one's protocol overlaps the other's burst.
    // The issuer count must divide every ring it indexes (TMEM stages, halo buffers): a ring slot is then always
    // handled by the same warp, in order - with slots shared between issuers a warp could test a barrier two phases
    // ahead, and mbarrier parity waits alias modulo 2.
    auto run_issuer = [&](auto ME_) {
      const int n_issuers = staged ? 1 : p.niss;   // warps 1, 3 (in this order); the launcher makes both rings multiples of it
      // `me` (which of the two issuers this warp is; a second issuer that is not needed simply finds no tile below) is a
      // COMPILE-TIME constant of each copy of this code: everything the MMA operands depend on (tile index, halo buffer, TMEM
      // stage) then derives from blockIdx / parameters / loop counters only, so ptxas keeps the descriptor arithmetic on the
      // uniform datapath. With `me` computed from the (shuffled) warp index it saw a divergent value and fed every UTCHMMA
      // through 6-8 R2UR.BROADCAST moves: ~80 cycles of issue per MMA against 44 cycles of pipe time (ncu: tensor pipe 35 %
      // active on the stems).
      constexpr int me = decltype(ME_)::value;
      // D = f32; A, B = bf16 (format 1) or fp16 (format 0, split-half mode), both K-major; N = NT; M = 128 / 256
      const uint32_t idesc = (1u << 4) | (p.f16 ? 0u : ((1u << 7) | (1u << 10))) | ((uint32_t)(p.NT >> 3) << 17) | ((uint32_t)((kPair ? 256 : 128) >> 4) << 24);
      int stage = 0;
      uint32_t phase = 0;
      long long t_wfull = 0, t_wtmem = 0, t_whalo = 0, t_begin = clock64();
      const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
      const uint32_t off_wres = halo ? (uint32_t)(p.a_bufs * p.a_bytes) : 0u;
      const uint32_t off_stages = off_wres + (p.resident ? (uint32_t)p.wres_bytes : 0u);
      if (p.resident) mbar_wait(wres_bar, 0, 6);
      if constexpr (NCLS > 1) {
        // ------------------------------------------------ fused deconv classes (the launcher guarantees two issuers)
        constexpr int CSH = NCLS == 4 ? 2 : 1;
        const int my_tiles = ((int)blockIdx.x < total_tiles) ? (total_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
        const int nv = my_tiles * NCLS;   // two issuers (the classes alternate by parity)
        const uint32_t a_lo = ((p.lbo_bytes >> 4) & 0x3FFF) << 16;
        const uint32_t a_hi = ((p.sbo_bytes >> 4) & 0x3FFF) | (1u << 14);
        const uint32_t b_hi128 = (1024u >> 4) | (1u << 14) | (2u << 29), b_hi64 = (512u >> 4) | (1u << 14) | (4u << 29);
        const uint32_t kstep16 = p.kstep_bytes >> 4;
        for (int v = me; v < nv; v += 2) {
          const int riter = v >> CSH, cls = v & (NCLS - 1);
          int as;
          uint32_t accphase;
          ring_of(v, acc_stages, p.acc_shift, as, accphase);
          long long tw = p.dbg ? clock64() : 0;
          mbar_wait(&tmem_empty[as], accphase ^ 1, 2);
          if (p.dbg) t_wtmem += clock64() - tw;
          int ab;
          uint32_t aph;
          ring_of(riter, p.a_bufs, p.a_shift, ab, aph);
          tw = p.dbg ? clock64() : 0;
          mbar_wait(&a_full[ab], aph, 7);
          if (p.dbg) t_whalo += clock64() - tw;
          tc_fence_after();
          const uint32_t tmem_d = tmem_base + as * acc_stride;
          const uint32_t sA = smem_base + (uint32_t)ab * p.a_bytes;
          const uint32_t sB = smem_base + off_wres + (uint32_t)cls * (uint32_t)p.cls_bytes;
          const uint32_t lead = elect_one() ? 1u : 0u;
          auto issue_cls = [&](auto CLS) {
            constexpr int C = decltype(CLS)::value;
            uint32_t acc = 0u;
  #pragma unroll
            for (int j = 0; j < R64; ++j) {
              const uint32_t a0 = (sA + p.aoff[C * C8_CLS_UNITS + j]) >> 4;
              const uint32_t b0 = (sB + j * b64_bytes) >> 4;
  #pragma unroll
              for (int k = 0; k < MMAS; ++k) {
                umma_bf16_if32(lead, tmem_d, a_lo | (a0 + k * kstep16), a_hi, b0 + 2 * k, b_hi128, idesc, acc);
                acc = 1u;
              }
            }
  #pragma unroll
            for (int j = 0; j < R32; ++j) {
              const uint32_t a0 = (sA + p.aoff[C * C8_CLS_UNITS + R64 + j]) >> 4;
              const uint32_t b0 = (sB + R64 * b64_bytes + j * b32_bytes) >> 4;
  #pragma unroll
              for (int k = 0; k < 2; ++k) {
                umma_bf16_if32(lead, tmem_d, a_lo | (a0 + k * kstep16), a_hi, b0 + 2 * k, b_hi64, idesc, acc);
                acc = 1u;
              }
            }
          };
          if (cls == 0) issue_cls(std::integral_constant<int, 0>{});
          else if (cls == 1) issue_cls(std::integral_constant<int, 1>{});
          else if (NCLS == 4 && cls == 2) issue_cls(std::integral_constant<int, NCLS == 4 ? 2 : 0>{});
          else issue_cls(std::integral_constant<int, NCLS == 4 ? 3 : 1>{});
          if (cls >= NCLS - 2) umma_commit_if(lead, &a_empty[ab]);   // this issuer's last class of the tile
          umma_commit_if(lead, &tmem_full[as]);
          __syncwarp();
        }
      } else {
      for (int iter = me, tile = (me < n_issuers) ? (int)(blockIdx.x + me * gridDim.x) : total_tiles; tile < total_tiles;
           tile += n_issuers * gridDim.x, iter += n_issuers) {
        int as;
        uint32_t accphase;
        ring_of(iter, acc_stages, p.acc_shift, as, accphase);
        long long tw = p.dbg ? clock64() : 0;
        if (kPair) mbar_wait_cluster(&tmem_empty[as], accphase ^ 1, 2); else mbar_wait(&tmem_empty[as], accphase ^ 1, 2);
        if (p.dbg) t_wtmem += clock64() - tw;
        C8_TRACE(iter, 1);
        int ab = 0;
        if (halo) {
          uint32_t aph;
          ring_of(iter, p.a_bufs, p.a_shift, ab, aph);
          tw = p.dbg ? clock64() : 0;
          mbar_wait(&a_full[ab], aph, 7);
          if (p.dbg) t_whalo += clock64() - tw;
        }
        C8_TRACE(iter, 2);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + as * acc_stride;
        for (int ks = 0; ks < (KS1 ? 1 : ksteps); ++ks) {
          if (staged) {
            tw = p.dbg ? clock64() : 0;
            mbar_wait(&full_bar[stage], phase, 3);
            if (p.dbg) t_wfull += clock64() - tw;
            tc_fence_after();
          }
          // shared-window addresses as plain 32-bit integer arithmetic on the (constant) window base: stays uniform
          const uint32_t st = smem_base + off_stages + (uint32_t)stage * stage_bytes;
          const uint32_t sB = p.resident ? smem_base + off_wres + (KS1 ? 0u : (uint32_t)ks * b_bytes) : st + stage_a;
          const uint32_t sA = halo ? smem_base + (uint32_t)ab * p.a_bytes : st;
          {
            const uint32_t lead = elect_one() ? 1u : 0u;   // predicate only: no divergent region around the issue loop
            uint32_t acc = (!KS1 && ks) ? 1u : 0u;
            // descriptors: only the 14-bit start-address field (bytes >> 4) changes between MMAs
            const uint32_t a_lo = ((p.lbo_bytes >> 4) & 0x3FFF) << 16;
            const uint32_t a_hi = ((p.sbo_bytes >> 4) & 0x3FFF) | (1u << 14);
            const uint32_t b_hi128 = (1024u >> 4) | (1u << 14) | (2u << 29), b_hi64 = (512u >> 4) | (1u << 14) | (4u << 29);
            const uint32_t kstep16 = p.kstep_bytes >> 4;
            const uint32_t n_u64 = p.ntaps * p.n64;
            // A offsets come from the constant bank (compile-time indices when the k-step structure is templated)
            const int u0 = KS1 ? 0 : ks * r64, v0 = KS1 ? R64 : (int)n_u64 + ks * r32;
  #pragma unroll
            for (int j = 0; j < (R64 >= 0 ? R64 : 32); ++j) {
              if (j < r64) {
                const uint32_t a0 = (sA + p.aoff[u0 + j]) >> 4;
                const uint32_t b0 = (sB + j * b64_bytes) >> 4;
  #pragma unroll
                for (int k = 0; k < 4; ++k) {
                  if (k < mmas64) {
                    if (kPair) umma2_bf16_if32(lead, tmem_d, a_lo | (a0 + k * kstep16), a_hi, b0 + 2 * k, b_hi128, idesc, acc);
                    else umma_bf16_if32(lead, tmem_d, a_lo | (a0 + k * kstep16), a_hi, b0 + 2 * k, b_hi128, idesc, acc);
                    acc = 1u;
                  }
                }
              }
            }
  #pragma unroll
            for (int j = 0; j < (R64 >= 0 ? R32 : 32); ++j) {
              if (j < r32) {
                const uint32_t a0 = (sA + p.aoff[v0 + j]) >> 4;
                const uint32_t b0 = (sB + r64 * b64_bytes + j * b32_bytes) >> 4;
  #pragma unroll
                for (int k = 0; k < 2; ++k) {
                  if (kPair) umma2_bf16_if32(lead, tmem_d, a_lo | (a0 + k * kstep16), a_hi, b0 + 2 * k, b_hi64, idesc, acc);
                  else umma_bf16_if32(lead, tmem_d, a_lo | (a0 + k * kstep16), a_hi, b0 + 2 * k, b_hi64, idesc, acc);
                  acc = 1u;
                }
              }
            }
            if (kPair) {
              if (staged) umma2_commit_if(lead, &empty_bar[stage]);
              if (KS1 || ks == ksteps - 1) {
                if (halo) umma2_commit_if(lead, &a_empty[ab]);
                umma2_commit_if(lead, &tmem_full[as]);
              }
            } else {
              if (staged) umma_commit_if(lead, &empty_bar[stage]);
              if (KS1 || ks == ksteps - 1) {
                if (halo) umma_commit_if(lead, &a_empty[ab]);
                umma_commit_if(lead, &tmem_full[as]);
              }
            }
          }
          __syncwarp();
          if (staged && ++stage == p.num_stages) { stage = 0; phase ^= 1; }
        }
        C8_TRACE(iter, 3);
      }
      }   // NCLS == 1

      if (p.dbg && lane == 0 && me == 0) { p.dbg[blockIdx.x * 8 + 2] = t_wfull; p.dbg[blockIdx.x * 8 + 3] = t_wtmem; p.dbg[blockIdx.x * 8 + 4] = clock64() - t_begin; p.dbg[blockIdx.x * 8 + 7] = t_whalo; }
    };
    if (warp == 1) run_issuer(std::integral_constant<int, 0>{});
    else run_issuer(std::integral_constant<int, 1>{});
  } else if (warp >= 4) {
    // ==================================================================== epilogue
    const int q = warp & 3;
    const int grp = (warp - 4) >> 2;
    const bool fast_epi = epi_fast_ok(p.e);
    const int row = q * 32 + lane;
    const int ry = row / C8_TW, rx = row % C8_TW;
    long long t_wacc = 0, t_begin = clock64();
    // tile-alternating groups (epi_split == 1) visit every TC_EPI_GROUPS-th tile of this CTA; a tile's coordinates
    // come from two unsigned divisions (cheaper than stepping the mixed-radix counter through the skipped tiles)
    // epi_split = 1 (N <= 128): the groups take alternate tiles, one or two TMEM stages each; epi_split = TC_EPI_GROUPS
    // (N = 192, two stages): all groups drain every tile together, group `sub` taking every epi_split-th column block
    const int nteams = TC_EPI_GROUPS / epi_split, team = grp / epi_split, sub = grp - team * epi_split;
    const int istep = nteams;
    const uint32_t tpi = (uint32_t)(p.tiles_x * p.tiles_y);
    // fused classes: `iter` counts VIRTUAL tiles (tile * NCLS + class); the launcher guarantees epi_split == 1 for them
    constexpr int CSH = NCLS == 4 ? 2 : (NCLS == 2 ? 1 : 0);
    for (int iter = team, tile = blockIdx.x + (iter >> CSH) * gridDim.x; tile < total_tiles;
         iter += istep, tile = blockIdx.x + (iter >> CSH) * gridDim.x) {
      const int cls = iter & (NCLS - 1);
      const uint32_t img_u = (uint32_t)tile / tpi, rem = (uint32_t)tile - img_u * tpi;
      const uint32_t ty_u = rem / (uint32_t)p.tiles_x;
      const int img = (int)img_u, ty = (int)ty_u, tx = (int)(rem - ty_u * (uint32_t)p.tiles_x);
      int as;
      uint32_t accphase;
      ring_of(iter, acc_stages, p.acc_shift, as, accphase);
      const long long tw = p.dbg ? clock64() : 0;
      mbar_wait(&tmem_full[as], accphase, 4);
      if (p.dbg) t_wacc += clock64() - tw;
      if (q == 0) C8_TRACE(iter, 4);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + as * acc_stride;
      const int py = ty * C8_TH + ry, px = tx * C8_TW + rx;
      const bool valid = (py < p.Ho) && (px < p.Wo);
      // output pixel of this position (sub-pixel classes: osy = osx = 2 and a per-class offset)
      const int oy = py * p.e.osy + (NCLS > 1 ? p.cls_ooy[cls] : p.e.ooy), ox = px * p.e.osx + (NCLS > 1 ? p.cls_oox[cls] : p.e.oox);
      if (p.e.nsplit > 1) {     // split-half output (fp32-on-tensor-cores mode): exact-math gate, hi / lo stores
        if (p.e.epi == EPI_GATE_ELU) tc_epilogue_gated_split<true>(p.e, bias_s, cst_n, taddr, img, valid, oy, ox, sub, epi_split);
        else tc_epilogue_gated_split<false>(p.e, bias_s, cst_n, taddr, img, valid, oy, ox, sub, epi_split);
      } else if (KS1 && p.ecst_nb) {   // (only the single-k-step instantiations carry this code: the launcher sets ecst_nb for them alone)
        // constants as kernel parameters (gated, bf16 block output, 2 or 3 blocks, one group per tile)
        const bool elu = (p.e.epi == EPI_GATE_ELU);
#ifdef SE_C8_TRACE
        unsigned long long* tr = (p.dbg && p.trace && blockIdx.x == 0 && iter < 64 && lane == 0 && q == 0) ? &p.dbg[2048 + iter * 8 + 7] : nullptr;
#else
        constexpr unsigned long long* tr = nullptr;
#endif
        if (p.ecst_nb == 3) { if (elu) tc_epilogue_gated_const<true, 3>(p.e, p.ecst, taddr, img, valid, oy, ox, tr); else tc_epilogue_gated_const<false, 3>(p.e, p.ecst, taddr, img, valid, oy, ox, tr); }
        else { if (elu) tc_epilogue_gated_const<true, 2>(p.e, p.ecst, taddr, img, valid, oy, ox, tr); else tc_epilogue_gated_const<false, 2>(p.e, p.ecst, taddr, img, valid, oy, ox, tr); }
      } else if (fast_epi) tc_epilogue_tile<true>(p.e, bias_s, cst_n, taddr, img, 0, valid, oy, ox, sub, epi_split);
      else tc_epilogue_tile<false>(p.e, bias_s, cst_n, taddr, img, 0, valid, oy, ox, sub, epi_split);
      if (q == 0) C8_TRACE(iter, 5);
      tc_fence_before();
      __syncwarp();
      // ONE arrival per warp: 128 per-thread arrivals on the same barrier are serialised shared-memory atomics, paid per tile
      if (lane == 0) {
        if (kPair) mbar_arrive_cluster(mapa_rank(smem_u32(&tmem_empty[as]), 0));   // the leader's MMA warp owns both accumulators
        else mbar_arrive(&tmem_empty[as]);
      }
      if (q == 0) C8_TRACE(iter, 6);
    }
    if (p.dbg && threadIdx.x == 128) { p.dbg[blockIdx.x * 8 + 5] = t_wacc; p.dbg[blockIdx.x * 8 + 6] = clock64() - t_begin; }
  }

  tc_fence_before();
  if (kPair) cluster_sync_all(); else __syncthreads();       // pair: no CTA may exit while its peer still reads its shared memory
  if (warp == 2) {
    tc_fence_after();
    if (kPair) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TC_TMEM_COLS) : "memory");
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TC_TMEM_COLS) : "memory");
  }
}

// ------------------------------------------------------------------------------------------ host
void fill_epi(const ConvParams& c, int NT, EpiParams* e) {
  e->y = c.y; e->out_dt = c.out_dt; e->out_c8 = c.out_c8;
  e->Hout = c.Hout; e->Wout = c.Wout; e->ldo = c.ldo; e->choff = c.choff;
  e->osy = c.osy; e->ooy = c.ooy; e->osx = c.osx; e->oox = c.oox;
  e->epi = c.epi; e->scale = c.scale; e->colscale = c.colscale;
  e->Cout = c.Cout; e->NT = NT;
  e->has_bias = c.bias != nullptr ? 1 : 0;
  e->blk_split = c.out_blk_split > 0 ? c.out_blk_split : (1 << 20);
  e->blk_jump = c.out_blk_split > 0 ? c.out_blk_jump : 0;
  e->par_stride = c.out_par_stride > 0 ? c.out_par_stride : (c.ldo >> 2);
  e->nsplit = c.f16x2 ? 2 : 1;
  e->split_stride = (int)c.out_split_stride;
  e->goff = (c.epi == EPI_LINEAR) ? 0 : gated_goff(c.Cout);
}
// the fast epilogue addresses the output in 32-bit units of 16 B
static inline bool epi_out_fits_u32(const ConvParams& c) {
  const double units = c.out_c8 ? (double)c.N * c.ldo * c.Hout * c.Wout : (double)c.N * c.Hout * c.Wout * c.ldo / 8.0;
  return units < 4294967296.0 && (reinterpret_cast<uintptr_t>(c.y) & 15) == 0;
}
bool epi_addressable(const ConvParams& c) { return epi_out_fits_u32(c); }

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn c8_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess || qres != cudaDriverEntryPointSuccess || !p) return nullptr;
    fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

static int g_sms = 0, g_optin = 0;
static const int kSmemBudget = 200 * 1024;
static const int kResidentMax = 112 * 1024;

// geometry shared by the weight packer (stage grouping) and the launcher
int c8_configure(C8Layer* L, int ntaps, const int8_t* dy, const int8_t* dx, int Ci, int Cout, bool stem, const int8_t* tap_cb) {
  L->stem = stem;
  int cb_max = 0;
  for (int t = 0; t < ntaps; ++t) {
    L->tap_cb[t] = tap_cb ? tap_cb[t] : 0;
    cb_max = L->tap_cb[t] > cb_max ? L->tap_cb[t] : cb_max;
  }
  int mn_y = 0, mx_y = 0, mn_x = 0, mx_x = 0;
  for (int t = 0; t < ntaps; ++t) {
    mn_y = dy[t] < mn_y ? dy[t] : mn_y; mx_y = dy[t] > mx_y ? dy[t] : mx_y;
    mn_x = dx[t] < mn_x ? dx[t] : mn_x; mx_x = dx[t] > mx_x ? dx[t] : mx_x;
  }
  const int extra_x = stem ? 5 : 0;   // the stem's GEMM-K walks 6 pixels to the right of the tap origin
  const int HR = C8_TH + (mx_y - mn_y), WR = C8_TW + (mx_x - mn_x) + extra_x;
  TcWeights& w = L->w;
  w.ntaps = ntaps;
  L->mmas64 = (stem || Ci == 48) ? 3 : 4;   // 48 channels = three K16 slices of the one 64-wide unit: the fourth would multiply padding
  if (stem) { w.n64 = 1; w.n32 = 0; }
  else {
    w.n64 = Ci / 64;
    int rem = Ci - 64 * w.n64;
    if (rem > 32) { ++w.n64; rem = 0; }
    w.n32 = rem > 0 ? 1 : 0;
  }
  // the box covers the zero-padded GEMM K (whole 64 / 32 channel chunks): blocks past the tensor are TMA zero fill,
  // so the MMAs never multiply stale shared memory (possibly NaN bit patterns) by the zero weight columns
  // (space-to-depth layers: a tap starts at its own channel block; the zero weight columns of its last chunk may then
  //  multiply the next parity's finite activations instead of TMA zeros, which is just as harmless)
  L->cb_in = stem ? 1 + cb_max : cb_max + (w.n64 * 64 + w.n32 * 32) / 8;   // (split-half stem input: hi block + lo block)
  const long long halo_bytes = (long long)L->cb_in * HR * WR * 16;
  w.NT = (gated_goff(Cout) + Cout / 2 + 15) / 16 * 16;   // every layer on this path is gated: gate columns start at goff
  w.n_tiles = 1;
  w.img_bytes = 0;
  const long long wbytes = (long long)ntaps * w.NT * (w.n64 * 128 + w.n32 * 64);
  // halo re-use while the region stays small enough to sit next to the weight stages (one or two buffers,
  // decided at launch); larger dilations fetch one box per tap
  L->mode = (halo_bytes <= 72 * 1024) ? C8_HALO : C8_PERTAP;
  if (L->mode == C8_HALO) {
    L->HR = HR; L->WR = WR; L->pad_y0 = -mn_y; L->pad_x0 = -mn_x;
  } else {
    L->HR = C8_TH; L->WR = C8_TW; L->pad_y0 = 0; L->pad_x0 = 0;
    L->cb_in = (w.n64 * 64 + w.n32 * 32) / 8;   // a box per tap, starting at the tap's own channel block (C8Params::tap_cb)
  }
  L->a_tx_bytes = L->cb_in * L->HR * L->WR * 16;
  L->a_bytes = (L->a_tx_bytes + 1023) / 1024 * 1024;
  L->resident = (wbytes <= kResidentMax) && (2 * L->a_bytes + wbytes <= kSmemBudget);
  // stage grouping: PERTAP -> one tap per stage; otherwise B-only stages of <= 48 KB (whole taps for mixed chunking)
  if (L->resident && L->mode == C8_HALO) {
    // nothing is streamed per k-step: one k-step issues every MMA of the tile back to back
    w.r64 = ntaps * w.n64;
    w.r32 = ntaps * w.n32;
  } else if (L->mode == C8_PERTAP || (w.n64 > 0 && w.n32 > 0)) { w.r64 = w.n64; w.r32 = w.n32; }
  else {
    const int unit = w.n64 ? w.NT * 128 : w.NT * 64, total = ntaps * (w.n64 ? w.n64 : w.n32);
    int best = 1;
    for (int k = 1; k <= 8 && k <= total; ++k)
      if (total % k == 0 && k * unit <= 48 * 1024) best = k;
    if (w.n64) { w.r64 = best; w.r32 = 0; } else { w.r64 = 0; w.r32 = best; }
  }
  if (L->mode == C8_PERTAP) SE_REQUIRE(tc_ksteps(w) == ntaps, "per-tap stages must be whole taps");
  return 0;
}

// the k-step structures of the generator's layers get their own fully unrolled instantiation
#define C8_SPECIALISATIONS(X) X(5, 0, 3) X(0, 9, 4) X(9, 0, 4) X(9, 0, 3) X(1, 0, 4) X(1, 0, 3) X(1, 1, 4) X(4, 4, 4) X(4, 0, 4) X(4, 0, 3) X(0, 3, 4) X(0, 1, 4) X(3, 0, 4) X(3, 0, 3)
// k-step structures of the streamed-weight layers that run as CTA pairs (96->192: <1,1>; 192/48->192: <1,0>;
// the 48->96 stride-2 layer of the refine branch: <3,0>)
#define C8_PAIR_SPECIALISATIONS(X) X(1, 0, 4) X(1, 0, 3) X(1, 1, 4) X(3, 0, 4) X(3, 0, 3)
// structures that occur with a single k-step per tile (resident weights): compile-time k-step index (KS1)
#define C8_KS1_SPECIALISATIONS(X) X(5, 0, 3) X(0, 9, 4) X(9, 0, 4) X(9, 0, 3) X(4, 4, 4) X(4, 0, 4) X(4, 0, 3)
// fused sub-pixel classes of the two deconv shapes: 48->48 (one 64-channel unit per tap, all 4 classes resident) and
// 96->96 (64 + 32 channel units per tap, 2 classes resident: one launch per output-row parity)
#define C8_GROUP_SPECIALISATIONS(X) X(4, 0, 4, 4) X(4, 0, 3, 4) X(4, 4, 4, 2) X(4, 0, 4, 2) X(4, 0, 3, 2) X(4, 4, 4, 4)
static int c8_set_smem_attr(int bytes) {
#define X(a, b, m) SE_CUDA_OK(cudaFuncSetAttribute(conv_c8_kernel<a, b, m, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  C8_SPECIALISATIONS(X)
#undef X
#define X(a, b, m) SE_CUDA_OK(cudaFuncSetAttribute(conv_c8_kernel<a, b, m, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  C8_PAIR_SPECIALISATIONS(X)
#undef X
#define X(a, b, m) SE_CUDA_OK(cudaFuncSetAttribute(conv_c8_kernel<a, b, m, 0, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  C8_KS1_SPECIALISATIONS(X)
#undef X
#define X(a, b, m, n) SE_CUDA_OK(cudaFuncSetAttribute(conv_c8_kernel<a, b, m, 0, 1, n>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  C8_GROUP_SPECIALISATIONS(X)
#undef X
  SE_CUDA_OK(cudaFuncSetAttribute(conv_c8_kernel<-1, 0, 0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  return 0;
}
static bool c8_pair_kernel_exists(int r64, int r32, int mmas64) {
#define X(a, b, m) if (r64 == a && r32 == b && mmas64 == m) return true;
  C8_PAIR_SPECIALISATIONS(X)
#undef X
  return false;
}
static int c8_dispatch(const C8Params& p, const CUtensorMap& tmA, const CUtensorMap& tmB, bool pair, int grid, int smem_bytes,
                       cudaStream_t stream) {
  if (pair) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(TC_NUM_THREADS); cfg.dynamicSmemBytes = smem_bytes; cfg.stream = stream;
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeClusterDimension;
    attr.val.clusterDim.x = 2; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
    cfg.attrs = &attr; cfg.numAttrs = 1;
#define X(a, b, m)                                                                             \
    if (p.r64 == a && p.r32 == b && p.mmas64 == m) {                                            \
      SE_CUDA_OK(cudaLaunchKernelEx(&cfg, conv_c8_kernel<a, b, m, 1>, tmA, tmB, p));            \
      return 0;                                                                                \
    }
    C8_PAIR_SPECIALISATIONS(X)
#undef X
    SE_REQUIRE(false, "no CTA-pair instantiation for this k-step structure");
  }
  if (p.ncls > 1) {
#define X(a, b, m, n)                                                                             \
    if (p.r64 == a && p.r32 == b && p.ncls == n && p.mmas64 == m) {                                \
      conv_c8_kernel<a, b, m, 0, 1, n><<<grid, TC_NUM_THREADS, smem_bytes, stream>>>(tmA, tmB, p); \
      return 0;                                                                                   \
    }
    C8_GROUP_SPECIALISATIONS(X)
#undef X
    SE_REQUIRE(false, "no fused-class instantiation for this k-step structure");
  }
  static const bool no_ks1 = getenv("SE_C8_NOKS1") != nullptr;   // A/B switch for experiments
  if (p.ksteps == 1 && p.resident && p.mode == C8_HALO && !no_ks1) {
#define X(a, b, m)                                                                             \
    if (p.r64 == a && p.r32 == b && (a == 0 || p.mmas64 == m)) {                               \
      conv_c8_kernel<a, b, m, 0, 1><<<grid, TC_NUM_THREADS, smem_bytes, stream>>>(tmA, tmB, p); \
      return 0;                                                                                \
    }
    C8_KS1_SPECIALISATIONS(X)
#undef X
  }
#define X(a, b, m)                                                                             \
  if (p.r64 == a && p.r32 == b && (a == 0 || p.mmas64 == m)) {                                 \
    conv_c8_kernel<a, b, m, 0><<<grid, TC_NUM_THREADS, smem_bytes, stream>>>(tmA, tmB, p);     \
    return 0;                                                                                  \
  }
  C8_SPECIALISATIONS(X)
#undef X
  conv_c8_kernel<-1, 0, 0, 0><<<grid, TC_NUM_THREADS, smem_bytes, stream>>>(tmA, tmB, p);
  return 0;
}

static const int kGroupSmemMax = 222 * 1024;   // fused classes may use (almost) the whole opt-in window: weights of all classes + 2 halos
static bool c8_group_kernel_exists(int r64, int r32, int ncls, int mmas64) {
#define X(a, b, m, n) if (r64 == a && r32 == b && ncls == n && mmas64 == m) return true;
  C8_GROUP_SPECIALISATIONS(X)
#undef X
  return false;
}

int c8_configure_group(C8Group* G, int ncls, int ntaps, const int8_t (*dy)[8], const int8_t (*dx)[8], const int* ooy, const int* oox, int Ci, int Cout) {
  static const bool off = getenv("SE_C8_NOGROUP") != nullptr;   // A/B switch for experiments
  if (off || ncls < 2 || ncls > C8_MAX_CLS || ntaps > 8) return 1;
  int mn_y = 0, mx_y = 0, mn_x = 0, mx_x = 0;
  for (int c = 0; c < ncls; ++c)
    for (int t = 0; t < ntaps; ++t) {
      mn_y = dy[c][t] < mn_y ? dy[c][t] : mn_y; mx_y = dy[c][t] > mx_y ? dy[c][t] : mx_y;
      mn_x = dx[c][t] < mn_x ? dx[c][t] : mn_x; mx_x = dx[c][t] > mx_x ? dx[c][t] : mx_x;
    }
  C8Layer& L = G->geo;
  L = C8Layer();
  TcWeights& w = L.w;
  w.ntaps = ntaps;
  w.n64 = Ci / 64;
  int rem = Ci - 64 * w.n64;
  if (rem > 32) { ++w.n64; rem = 0; }
  w.n32 = rem > 0 ? 1 : 0;
  w.NT = (gated_goff(Cout) + Cout / 2 + 15) / 16 * 16;
  w.n_tiles = 1;
  w.img_bytes = 0;
  w.r64 = ntaps * w.n64;      // resident weights + halo: one k-step issues every MMA of a (tile, class)
  w.r32 = ntaps * w.n32;
  L.mmas64 = Ci == 48 ? 3 : 4;
  if (w.r64 + w.r32 > C8_CLS_UNITS || !c8_group_kernel_exists(w.r64, w.r32, ncls, L.mmas64)) return 1;
  L.mode = C8_HALO;
  L.resident = true;
  L.stem = false;
  L.cb_in = (w.n64 * 64 + w.n32 * 32) / 8;
  L.HR = C8_TH + (mx_y - mn_y); L.WR = C8_TW + (mx_x - mn_x);
  L.pad_y0 = -mn_y; L.pad_x0 = -mn_x;
  L.a_tx_bytes = L.cb_in * L.HR * L.WR * 16;
  L.a_bytes = (L.a_tx_bytes + 1023) / 1024 * 1024;
  G->ncls = ncls;
  G->ntaps = ntaps;
  G->cls_bytes = ntaps * w.NT * (w.n64 * 128 + w.n32 * 64);
  for (int c = 0; c < ncls; ++c) {
    for (int t = 0; t < ntaps; ++t) { G->dy[c][t] = dy[c][t]; G->dx[c][t] = dx[c][t]; }
    G->ooy[c] = ooy[c]; G->oox[c] = oox[c];
  }
  // weights of all classes + two halo buffers + barriers / constants must fit the opt-in window
  if (1024 + ncls * G->cls_bytes + 2 * L.a_bytes + 4096 > kGroupSmemMax) return 1;
  return 0;
}

// may this layer run as CTA pairs? (decided at packing time: the pair-format weight image is built only then)
bool c8_pair_capable(const C8Layer& L) {
  static const bool off = getenv("SE_C8_NOPAIR") != nullptr;
  const TcWeights& w = L.w;
  if (off || L.resident || L.stem || w.NT % 32 != 0) return false;
  const int half_bytes = (w.NT / 2) * (w.r64 * 128 + w.r32 * 64);
  return half_bytes % 512 == 0 && c8_pair_kernel_exists(w.n64 ? w.r64 : 0, w.n32 ? w.r32 : 0, L.mmas64);
}

int c8_launch(const ConvParams& c, const C8Layer& L_in, cudaStream_t stream, const C8Group* grp) {
  const C8Layer& L = grp ? grp->geo : L_in;
  const TcWeights& w = L.w;
  SE_REQUIRE((c.in_dt == DT_BF16 || c.in_dt == DT_F16X2) && c.in_c8 == 1, "conv_c8 reads 16-bit channel-blocked activations");
  SE_REQUIRE((c.in_dt == DT_F16X2) == (c.f16x2 != 0) && (c.out_dt == DT_F16X2) == (c.f16x2 != 0), "split-half mode: both sides");
  SE_REQUIRE(c.stride == 1, "conv_c8 handles stride-1 convolutions");
  SE_REQUIRE((reinterpret_cast<uintptr_t>(c.x) & 127) == 0, "input base must be 128 B aligned");
  SE_REQUIRE(c.ntaps == w.ntaps && c.ntaps <= MAX_TAPS, "tap count mismatch");
  for (int t = 0; t < c.ntaps && !grp; ++t) SE_REQUIRE(c.tap_cb[t] == L.tap_cb[t], "per-tap channel blocks differ from the packed layer");
  SE_REQUIRE(c.Wi * 8 <= (1 << 30) && L.WR * 8 <= 256 && L.HR <= 256 && L.cb_in <= 256, "TMA box limits");
  C8Params p;
  memset(&p, 0, sizeof(p));
  p.f16 = c.f16x2 ? 1 : 0;
  for (int t = 0; t < c.ntaps; ++t) p.tap_cb[t] = L.tap_cb[t];
  p.N = c.N; p.Ho = c.Ho; p.Wo = c.Wo;
  p.tiles_x = (c.Wo + C8_TW - 1) / C8_TW;
  p.tiles_y = (c.Ho + C8_TH - 1) / C8_TH;
  p.ntaps = c.ntaps;
  memcpy(p.dy, c.dy, sizeof(p.dy));
  memcpy(p.dx, c.dx, sizeof(p.dx));
  p.n64 = w.n64; p.n32 = w.n32; p.r64 = w.n64 ? w.r64 : 0; p.r32 = w.n32 ? w.r32 : 0; p.NT = w.NT;
  p.ksteps = tc_ksteps(w);
  p.w = reinterpret_cast<const uint8_t*>(grp ? grp->w_all : w.data);
  p.mode = L.mode; p.HR = L.HR; p.WR = L.WR; p.pad_y0 = L.pad_y0; p.pad_x0 = L.pad_x0;
  p.cb_in = L.cb_in; p.x_cb_off = c.x_cb_off;
  p.a_bytes = L.a_bytes; p.a_tx_bytes = L.a_tx_bytes;
  p.resident = L.resident ? 1 : 0;
  p.wres_bytes = grp ? grp->ncls * grp->cls_bytes : (int)tc_weight_bytes_per_image(w);
  p.ncls = grp ? grp->ncls : 1;
  p.cls_bytes = grp ? grp->cls_bytes : 0;
  for (int k = 0; k < C8_MAX_CLS; ++k) { p.cls_ooy[k] = grp && k < grp->ncls ? grp->ooy[k] : 0; p.cls_oox[k] = grp && k < grp->ncls ? grp->oox[k] : 0; }
  if (L.stem) { p.lbo_bytes = 16; p.kstep_bytes = 32; p.mmas64 = 3; }
  else { p.lbo_bytes = L.HR * L.WR * 16; p.kstep_bytes = 2 * p.lbo_bytes; p.mmas64 = L.mmas64; }
  p.sbo_bytes = L.WR * 16;
  p.bias = c.bias;
  fill_epi(c, w.NT, &p.e);
  SE_REQUIRE(c.out_dt == DT_F32 || epi_addressable(c), "output tensor too large / misaligned for 32-bit block addressing");
  {
    // epilogue constants as kernel parameters when the tile is drained by one group and has 2 or 3 blocks (N <= 48: the
    // 256^2 / 128^2 layers; with 6 blocks the two-pass form measured slower than the shared-memory constants)
    static const bool no_ecst = getenv("SE_C8_NOECST") != nullptr;   // A/B switch for experiments
    const int half = c.Cout / 2, nb = (half + 7) / 8;
    p.ecst_nb = 0;
    if (!no_ecst && !c.f16x2 && c.epi != EPI_LINEAR && c.bias_host != nullptr && epi_fast_ok(p.e) && w.NT <= 128 && (nb == 2 || nb == 3) &&
        tc_ksteps(w) == 1 && L.resident && L.mode == C8_HALO) {
      p.ecst_nb = nb;
      for (int i = 0; i < 24; ++i) {
        const float bf = i < half ? c.bias_host[i] : 0.0f, bg = i < half ? c.bias_host[half + i] : 0.0f;
        p.ecst[0][i] = bf;
        p.ecst[1][i] = bf * 1.4426950408889634f;
        p.ecst[2][i] = 0.5f * bg;
      }
    }
  }
  {
    // A-operand byte offsets inside the shared-memory region, per K unit (tile independent):
    // 64-wide units first (u = tap*n64 + chunk), then the 32-wide unit of each tap
    const bool halo = (L.mode == C8_HALO);
    const int n_u64 = c.ntaps * w.n64, n_u32 = c.ntaps * w.n32;
    SE_REQUIRE(n_u64 + n_u32 < C8_MAX_UNITS, "too many K units");
    SE_REQUIRE(!grp || n_u64 + n_u32 <= C8_CLS_UNITS, "too many K units per class");
    for (int k = 0; k < (grp ? grp->ncls : 1); ++k)
      for (int u = 0; u < n_u64 + n_u32; ++u) {
        const bool is64 = u < n_u64;
        const int t = is64 ? u / w.n64 : u - n_u64;
        const int cb0 = (halo ? L.tap_cb[t] : 0) + (is64 ? (u - t * w.n64) * 8 : w.n64 * 8);   // PERTAP: the box starts at the tap's block
        const int tdy = grp ? grp->dy[k][t] : c.dy[t], tdx = grp ? grp->dx[k][t] : c.dx[t];
        const int oy = halo ? tdy + L.pad_y0 : 0, ox = halo ? tdx + L.pad_x0 : 0;
        p.aoff[k * C8_CLS_UNITS + u] = (uint32_t)((cb0 * L.HR + oy) * L.WR + ox) * 16u;
      }
  }
  SE_REQUIRE(c.epi == EPI_LINEAR || (c.Cout % 2 == 0 && (c.out_dt == DT_BF16 || c.out_dt == DT_F16X2)), "gated epilogue needs even Cout, 16-bit out");
  SE_REQUIRE(!c.out_c8 || ((c.out_dt == DT_BF16 || c.out_dt == DT_F16X2) && c.choff % 8 == 0), "C8 output must be 16-bit with a channel offset multiple of 8");
  SE_REQUIRE(!c.f16x2 || (c.out_c8 != 0 && c.epi != EPI_LINEAR), "split-half output is channel-blocked and gated");
  SE_REQUIRE(c.out_c8 != 2 || (c.epi != EPI_LINEAR && c.Hout % 2 == 0 && c.Wout % 2 == 0 && c.ldo % 4 == 0 && (c.Cout / 2) % 8 == 0),
             "space-to-depth output: gated layer, even size, whole channel blocks");

  const int total_tiles = p.N * p.tiles_x * p.tiles_y;
  const bool pair = !grp && L.w_pair != nullptr && total_tiles % 2 == 0;
  const int smem_budget = grp ? kGroupSmemMax - 4096 : kSmemBudget;
  const int b_bytes = pair ? tc_stage_b_bytes(w) / 2 : tc_stage_b_bytes(w);   // per CTA
  const int stage_bytes = (L.mode == C8_HALO ? 0 : L.a_bytes) + (L.resident ? 0 : b_bytes);
  int fixed = (L.resident ? p.wres_bytes : 0);
  // ---- rings and MMA issuers. Every ring is a power of two (the kernel indexes them with a mask and a shift). A resident layer
  // with nothing streamed per k-step issues one short burst of MMAs per tile, so two issuer warps (1 and 3) take alternate tiles
  // when its halo ring is even: an issuer count must divide every ring it indexes, so that a slot is always handled by the same
  // warp, in order
  p.a_bufs = 2;
  p.niss = 1;
  p.acc_stages = w.NT <= 64 ? 8 : (w.NT <= 128 ? 4 : 2);
  p.acc_stride = w.NT <= 64 ? 64 : (w.NT <= 128 ? 128 : 256);
  // groups per tile (see the epilogue loop): one for N <= 128, all of them for wider tiles
  p.epi_split = w.NT <= 128 ? 1 : TC_EPI_GROUPS;
  SE_REQUIRE(p.epi_split == 1 || c.f16x2 || c.epi == EPI_LINEAR || !epi_fast_ok(p.e) || (c.Cout / 2 + 7) / 8 == 3 * p.epi_split,
             "a column-split fast gated epilogue needs three 8-column blocks per group");
  if (L.mode == C8_HALO) {
    if (fixed + 2 * L.a_bytes + 3 * stage_bytes > smem_budget) p.a_bufs = 1;   // measured: 2 halo buffers + 3 weight stages beats 1 + 4
    // nothing streamed: a tile is short (700-2000 cycles of MMAs) against a TMA round trip of ~1500 cycles, so two
    // halo buffers leave the tensor pipe waiting for loads; ring as deep as shared memory allows
    if (stage_bytes == 0) {
      while (p.a_bufs < C8_MAX_ABUFS && fixed + 2 * p.a_bufs * L.a_bytes <= smem_budget) p.a_bufs *= 2;
      p.niss = p.a_bufs % 2 == 0 ? 2 : 1;
    }
    fixed += p.a_bufs * L.a_bytes;
  }
  p.a_shift = -1;
  for (int sh = 0; sh < 4; ++sh) if ((1 << sh) == p.a_bufs) p.a_shift = sh;
  p.acc_shift = -1;
  for (int sh = 0; sh < 4; ++sh) if ((1 << sh) == p.acc_stages) p.acc_shift = sh;
  SE_REQUIRE(p.a_shift >= 0 && p.acc_shift >= 0 && p.acc_stages * p.acc_stride <= TC_TMEM_COLS && p.a_bufs <= C8_MAX_ABUFS &&
                 p.a_bufs % p.niss == 0 && p.acc_stages % p.niss == 0,
             "ring / issuer plan");
  SE_REQUIRE(!grp || (p.a_bufs >= 2 && w.NT <= 128 && p.ksteps == 1), "fused classes need two halo buffers, <= 128 accumulator columns and a single k-step");
  int stages = stage_bytes ? (smem_budget - fixed) / stage_bytes : 1;
  if (stages > TC_MAX_STAGES) stages = TC_MAX_STAGES;
  SE_REQUIRE(stages >= (stage_bytes ? 2 : 1), "shared memory plan does not fit");
  p.num_stages = stages;
  const int smem_bytes = 1024 + fixed + stages * stage_bytes + (2 * TC_MAX_STAGES + 2 * C8_MAX_ABUFS + 17) * 8 + 16 + 3 * (p.NT + 32) * 4 + 64;

  EncodeTiledFn enc = c8_encode_fn();
  SE_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled not available from the driver");
  if (!g_sms) {
    int dev = 0;
    SE_CUDA_OK(cudaGetDevice(&dev));
    SE_CUDA_OK(cudaDeviceGetAttribute(&g_sms, cudaDevAttrMultiProcessorCount, dev));
    SE_CUDA_OK(cudaDeviceGetAttribute(&g_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    { int rc_attr = c8_set_smem_attr(g_optin); if (rc_attr) return rc_attr; }
  }
  SE_REQUIRE(smem_bytes <= g_optin, "shared memory plan exceeds the opt-in limit");

  CUtensorMap tmA;
  {
    // C8 activations viewed as (8*W, H, CB, N): a row of the box is WR pixels x 16 B, contiguous in memory
    cuuint64_t dims[4] = {(cuuint64_t)c.Wi * 8, (cuuint64_t)c.Hi, (cuuint64_t)c.ldx, (cuuint64_t)c.N};
    cuuint64_t strides[3] = {(cuuint64_t)c.Wi * 16, (cuuint64_t)c.Hi * c.Wi * 16, (cuuint64_t)c.ldx * c.Hi * c.Wi * 16};
    cuuint32_t box[4] = {(cuuint32_t)(L.WR * 8), (cuuint32_t)L.HR, (cuuint32_t)L.cb_in, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(&tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(c.x), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    SE_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(C8) failed, CUresult=" + std::to_string((int)r));
  }
  CUtensorMap tmB;
  memset(&tmB, 0, sizeof(tmB));
  if (pair) {
    // pair-format weights viewed as 512 B rows (the longest a box row can be: fewest TMA row requests):
    // stage ks = [rank 0 half][rank 1 half], one box per (stage, rank)
    SE_REQUIRE(b_bytes % 512 == 0 && b_bytes / 512 <= 256, "pair weight stage must be whole 512 B rows");
    const int rows_half = b_bytes / 512;
    cuuint64_t dims[2] = {256, (cuuint64_t)p.ksteps * 2 * rows_half};
    cuuint64_t strides[1] = {512};
    cuuint32_t box[2] = {256, (cuuint32_t)rows_half};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(&tmB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(L.w_pair), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    SE_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(pair weights) failed, CUresult=" + std::to_string((int)r));
  }
  int grid = total_tiles < g_sms ? total_tiles : g_sms;
  if (pair) grid &= ~1;
  p.step_x = grid % p.tiles_x;
  p.step_y = (grid / p.tiles_x) % p.tiles_y;
  p.step_img = grid / (p.tiles_x * p.tiles_y);
  static const bool dbg_on = getenv("SE_TC_DEBUG") != nullptr;
  static unsigned long long* dbg_buf = nullptr;
  if (dbg_on) {
    if (!dbg_buf) SE_CUDA_OK(cudaMalloc(&dbg_buf, 8 * 4096));
    SE_CUDA_OK(cudaMemsetAsync(dbg_buf, 0, 8 * 4096, stream));
    p.dbg = dbg_buf;
#ifdef SE_C8_TRACE
    p.trace = atoi(getenv("SE_TC_DEBUG")) >= 2 ? 1 : 0;
#else
    p.trace = 0;
#endif
  }
  { int rc_launch = c8_dispatch(p, tmA, tmB, pair, grid, smem_bytes, stream); if (rc_launch) return rc_launch; }
  SE_CUDA_OK(cudaGetLastError());
  if (dbg_on) {
    SE_CUDA_OK(cudaStreamSynchronize(stream));
    std::vector<unsigned long long> h(8 * grid);
    SE_CUDA_OK(cudaMemcpy(h.data(), dbg_buf, h.size() * 8, cudaMemcpyDeviceToHost));
    double a[8] = {0};
    for (int b = 0; b < grid; ++b)
      for (int k = 0; k < 8; ++k) a[k] += (double)h[b * 8 + k] / grid;
    fprintf(stderr,
            "[c8] N=%d %dx%d Ci=%d taps=%d NT=%d mode=%s pair=%d res=%d HRxWR=%dx%d abufs=%d n64=%d n32=%d r64=%d r32=%d stages=%d tiles=%d | prod wait %.0f/%.0f | mma wait_full %.0f wait_halo %.0f wait_tmem %.0f /%.0f | epi wait_acc %.0f/%.0f\n",
            c.N, c.Ho, c.Wo, c.Ci, c.ntaps, p.NT, L.mode == C8_HALO ? "halo" : "pertap", (int)pair, p.resident, L.HR, L.WR, p.a_bufs, p.n64, p.n32, p.r64, p.r32,
            p.num_stages, total_tiles, a[0], a[1], a[2], a[7], a[3], a[4], a[5], a[6]);
    if (p.trace) {
      std::vector<unsigned long long> t(64 * 8);
      SE_CUDA_OK(cudaMemcpy(t.data(), dbg_buf + 2048, t.size() * 8, cudaMemcpyDeviceToHost));
      unsigned long long t0 = ~0ull;
      for (auto v : t) if (v && v < t0) t0 = v;
      fprintf(stderr, "[c8 trace] CTA 0, cycles since its first event: iter | tma_issued | got_tmem got_halo mma_issued | acc_seen epi_done released | tmem_loaded   (acc_stages=%d niss=%d abufs=%d)\n",
              p.acc_stages, p.niss, p.a_bufs);
      for (int i = 0; i < 64 && i * (int)(grid) < total_tiles; ++i) {
        fprintf(stderr, "[c8 trace] %2d |", i);
        for (int k = 0; k < 8; ++k) fprintf(stderr, " %7lld%s", t[i * 8 + k] ? (long long)(t[i * 8 + k] - t0) : -1LL, (k == 0 || k == 3 || k == 6) ? " |" : "");
        fprintf(stderr, "\n");
      }
    }
  }
  return 0;
}

}  // namespace se
