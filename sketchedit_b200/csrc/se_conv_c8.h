// Host/device interface of the channel-blocked tcgen05 convolution (se_conv_c8.cu).
#pragma once
#include "se_common.cuh"
#include "se_conv_tc.h"

namespace se {

enum { C8_HALO = 0, C8_PERTAP = 1 };
constexpr int C8_MAX_ABUFS = 8;   // halo ring depth (resident layers)
constexpr int C8_MAX_UNITS = 128;   // (tap, channel chunk) K units per tile (split-half layers: 3 products per tap)

// per-layer (per sub-pixel class) configuration fixed at weight-packing time
struct C8Layer {
  TcWeights w;          // B stage images (se_conv_tc.h), n_tiles = 1, shared weights
  int mode = C8_HALO;
  bool resident = false;
  bool stem = false;    // GEMM-K walks the pixel window of the 8-channel packed input
  int cb_in = 0;        // channel blocks read
  int mmas64 = 4;       // K16 MMAs per 64-channel unit: 3 when the layer has 48 input channels (the unit's last 16 are padding), 3 for stems
  int HR = 0, WR = 0;   // rows / columns of the shared-memory A region
  int pad_y0 = 0, pad_x0 = 0;
  int a_bytes = 0, a_tx_bytes = 0;
  int8_t tap_cb[MAX_TAPS] = {0};   // first channel block read by each tap (0 except space-to-depth layers)
  const void* w_pair = nullptr;   // CTA-pair format of the stage images (each stage = [rows 0..NT/2) | rows NT/2..NT)), or null
};

// Sub-pixel classes of one x2 deconv layer fused into ONE launch ("virtual tiles" = tile x class): the union halo of the
// classes' 2x2 windows is loaded once per tile, the resident weights of all classes sit in shared memory back to back,
// every (tile, class) gets its own TMEM stage / epilogue group, and the classes' interleaved output pixels are written
// from one SM within microseconds of each other (whole sectors reach DRAM instead of 16 B slivers per launch).
constexpr int C8_MAX_CLS = 4;
constexpr int C8_CLS_UNITS = 16;   // aoff[] stride per class
struct C8Group {
  C8Layer geo;                    // union-halo geometry; geo.w = the per-class stage structure (identical for all classes)
  int ncls = 0;
  int ntaps = 0;
  int8_t dy[C8_MAX_CLS][8], dx[C8_MAX_CLS][8];
  int ooy[C8_MAX_CLS], oox[C8_MAX_CLS];
  int cls_bytes = 0;              // resident weight image of one class
  const void* w_all = nullptr;    // device: ncls class images back to back
};

struct C8Params {
  int N, Ho, Wo;
  int tiles_x, tiles_y;
  int step_x, step_y, step_img;   // gridDim.x decomposed in (tiles_x, tiles_y, images): incremental tile decode
  int ntaps;
  int8_t dy[MAX_TAPS], dx[MAX_TAPS];
  int n64, n32, r64, r32, NT, ksteps;
  const uint8_t* w;
  int mode, HR, WR, pad_y0, pad_x0, cb_in, x_cb_off;
  int a_bytes, a_tx_bytes, a_bufs, a_shift;   // halo ring: a_bufs buffers (a power of two), a_shift = log2(a_bufs)
  int acc_stages, acc_shift, acc_stride;      // TMEM accumulator ring (same convention), columns between stages
  int epi_split;                              // 1: the epilogue groups take alternate tiles; 4: they split the columns of every tile
  int niss;                                   // MMA issuer warps (1 or 2); must divide both rings
  int lbo_bytes, sbo_bytes, kstep_bytes, mmas64;
  uint32_t aoff[C8_MAX_UNITS];   // byte offset of each K unit's A operand inside the shared-memory region
  int num_stages, resident, wres_bytes;
  const float* bias;
  EpiParams e;
  // gated layers with <= 24 outputs (the N <= 48 layers at 256^2 / 128^2): epilogue constants by accumulator column as kernel parameters,
  // [0] bias of feature c, [1] bias * log2(e), [2] 0.5 * bias of gate c; with a compile-time column count they become
  // constant-bank operands of the FMAs (no shared-memory loads in the epilogue). ecst_nb = 8-column blocks, 0 = unused
  int ecst_nb;
  float ecst[3][24];
  int f16;                        // operands are fp16 (split-half mode) instead of bf16
  int8_t tap_cb[MAX_TAPS];        // PERTAP mode: first channel block of each tap's box (split-half / space-to-depth inputs)
  int ncls, cls_bytes;            // fused deconv classes (C8Group): classes per tile, bytes between their weight images
  int cls_ooy[C8_MAX_CLS], cls_oox[C8_MAX_CLS];
  unsigned long long* dbg;
  int trace;   // SE_TC_DEBUG=2: per-tile timeline of CTA 0 (C8_TRACE)
};

int c8_configure(C8Layer* L, int ntaps, const int8_t* dy, const int8_t* dx, int Ci, int Cout, bool stem, const int8_t* tap_cb = nullptr);
bool c8_pair_capable(const C8Layer& L);
// byte offset of element (unit, n, k) of a stage in the CTA-pair image: the two row halves are separate sub-images
inline uint32_t c8_pair_image_offset(const TcWeights& w, bool is64, int j, int n, int k) {
  const int NTh = w.NT / 2;
  const uint32_t half_bytes = (uint32_t)NTh * (w.r64 * 128 + w.r32 * 64);
  return (uint32_t)(n / NTh) * half_bytes + tc_b_image_offset(NTh, w.n64 ? w.r64 : 0, is64, j, n % NTh, k);
}
int c8_launch(const ConvParams& c, const C8Layer& L, cudaStream_t stream, const C8Group* grp = nullptr);
// geometry of a fused-class launch; returns non-zero (no error text) when the classes do not fit in shared memory
int c8_configure_group(C8Group* G, int ncls, int ntaps, const int8_t (*dy)[8], const int8_t (*dx)[8], const int* ooy, const int* oox, int Ci, int Cout);

}  // namespace se
