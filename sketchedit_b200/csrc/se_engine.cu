// Host side of the library: weight packing, the generator forward graph, the C ABI
// (include/sketchedit_b200.h). Graph structure follows
//   MDGenerator.forward            reference models/networks/editline2_g.py:59-94
//   DeepFillC2Generator.forward    reference models/networks/editline_g.py:119-221
//   EditLine2Model inference       reference models/editline2_model.py:128-133,338-370
#include <stdlib.h>

#include <cuda_fp16.h>

#include <algorithm>
#include <cmath>
#include <functional>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/sketchedit_b200.h"
#include "se_common.cuh"
#include "se_conv_direct.h"
#include "se_conv_c8.h"
#include "se_cam.h"
#include "se_gemm_split.h"
#include "se_conv_tc.h"
#include "se_misc.h"
#include "se_resize.h"

namespace se {

static thread_local std::string g_err;
void set_error(const std::string& msg) { g_err = msg; }
const char* last_error() { return g_err.c_str(); }

static thread_local int g_launches = 0;

// ------------------------------------------------------------------------------------------ launch timing
// se_timing_enable(1): every launch of a forward is bracketed by CUDA events on its stream and accounted to a kernel
// class (kernel + layer shape) together with its ALGORITHMIC work: 2*MAC of the reference op (SURVEY.md 8d), the MACs
// this implementation really issues (sub-pixel deconvs: 4/9 of the reference's), and the bytes the op must move (input
// once, output once, weights once). bench.py runs ONE instrumented pass for the roofline table; the throughput passes
// run with timing off. Process-wide, guarded by a mutex.
struct TimedLaunch { cudaEvent_t a, b; int cls; };
struct ClassAgg { std::string name; int tensor; double flops_alg, flops_exec, bytes_alg; int launches; double ms; };
static std::mutex g_time_mu;
static bool g_timing = false;
static std::vector<TimedLaunch> g_tl;
static size_t g_tl_used = 0;
static std::vector<ClassAgg> g_classes;
static std::map<std::string, int> g_class_idx;

struct LaunchTag {
  std::string name;
  int tensor = 0;
  double flops_alg = 0, flops_exec = 0, bytes_alg = 0;
  bool set = false;
};

static int timing_begin(const LaunchTag& t, cudaStream_t st, size_t* slot) {
  std::lock_guard<std::mutex> lk(g_time_mu);
  const std::string key = t.set ? t.name : std::string("other");
  auto it = g_class_idx.find(key);
  int ci;
  if (it == g_class_idx.end()) {
    ci = (int)g_classes.size();
    g_class_idx[key] = ci;
    g_classes.push_back(ClassAgg{key, t.tensor, 0, 0, 0, 0, 0});
  } else ci = it->second;
  ClassAgg& a = g_classes[ci];
  a.flops_alg += t.flops_alg; a.flops_exec += t.flops_exec; a.bytes_alg += t.bytes_alg; a.launches += 1;
  if (g_tl_used == g_tl.size()) {
    TimedLaunch tl;
    SE_CUDA_OK(cudaEventCreate(&tl.a));
    SE_CUDA_OK(cudaEventCreate(&tl.b));
    g_tl.push_back(tl);
  }
  *slot = g_tl_used++;
  g_tl[*slot].cls = ci;
  SE_CUDA_OK(cudaEventRecord(g_tl[*slot].a, st));
  return 0;
}
static int timing_end(size_t slot, cudaStream_t st) {
  std::lock_guard<std::mutex> lk(g_time_mu);
  SE_CUDA_OK(cudaEventRecord(g_tl[slot].b, st));
  return 0;
}

// ------------------------------------------------------------------------------------------ architecture
struct Spec {
  const char* name;
  int cin, cout, k, stride, rate;
  bool deconv;
  int act;   // 0 elu, 1 relu, -1 none
};

static std::vector<Spec> encoder(const std::string& pfx, int cin0, std::vector<std::string>& names) {
  const int c = 48;
  struct R { const char* n; int ci, co, k, s, r; };
  const R rows[10] = {{"conv1", cin0, c, 5, 1, 1},          {"conv2_downsample", c / 2, 2 * c, 3, 2, 1},
                      {"conv3", c, 2 * c, 3, 1, 1},         {"conv4_downsample", c, 4 * c, 3, 2, 1},
                      {"conv5", 2 * c, 4 * c, 3, 1, 1},     {"conv6", 2 * c, 4 * c, 3, 1, 1},
                      {"conv7_atrous", 2 * c, 4 * c, 3, 1, 2},  {"conv8_atrous", 2 * c, 4 * c, 3, 1, 4},
                      {"conv9_atrous", 2 * c, 4 * c, 3, 1, 8},  {"conv10_atrous", 2 * c, 4 * c, 3, 1, 16}};
  std::vector<Spec> v;
  for (auto& r : rows) {
    names.push_back(pfx + r.n);
    v.push_back(Spec{nullptr, r.ci, r.co, r.k, r.s, r.r, false, 0});
  }
  return v;
}

struct ArchTable {
  std::vector<std::string> names;
  std::vector<Spec> specs;
  void add(const std::string& n, int ci, int co, int k = 3, int s = 1, int r = 1, bool deconv = false, int act = 0) {
    if (co == 3) act = -1;   // reference utils.py:27
    names.push_back(n);
    specs.push_back(Spec{nullptr, ci, co, k, s, r, deconv, act});
  }
  void add_encoder(const std::string& pfx, int cin0) {
    std::vector<std::string> nn;
    auto v = encoder(pfx, cin0, nn);
    for (size_t i = 0; i < v.size(); ++i) { names.push_back(nn[i]); specs.push_back(v[i]); }
  }
  void add_decoder(const std::string& pfx, int cin11, int cout17) {
    const int c = 48;
    add(pfx + "11", cin11, 4 * c);
    add(pfx + "12", 2 * c, 4 * c);
    add(pfx + "13_upsample_conv", 2 * c, 2 * c, 3, 1, 1, true);
    add(pfx + "14", c, 2 * c);
    add(pfx + "15_upsample_conv", c, c, 3, 1, 1, true);
    add(pfx + "16", c / 2, c / 2);
    add(pfx + "17", c / 4, cout17, 3, 1, 1, false, -1);
  }
};

static ArchTable make_arch(char net) {
  ArchTable t;
  const int c = 48;
  if (net == 'M') {
    t.add_encoder("", 4);
    t.add_decoder("conv", 2 * c, 3);
    t.add_decoder("conv_mask_", 2 * c, 1);
  } else {
    t.add_encoder("", 5);
    t.add_decoder("conv", 4 * c, 3);
    t.add_encoder("w", 5);
    t.add("xconv1", 3, c, 5);
    t.add("xconv2_downsample", c / 2, c, 3, 2);
    t.add("xconv3", c / 2, 2 * c);
    t.add("xconv4_downsample", c, 2 * c, 3, 2);
    t.add("xconv5", c, 4 * c);
    t.add("xconv6", 2 * c, 4 * c);
    t.add("xconv7_atrous", 2 * c, 4 * c, 3, 1, 2);
    t.add("xconv8_atrous", 2 * c, 4 * c, 3, 1, 4);
    t.add("xconv9_atrous", 2 * c, 4 * c, 3, 1, 8);
    t.add("xconv10_atrous", 2 * c, 4 * c, 3, 1, 16);
    t.add("pmconv1", 3, c, 5);
    t.add("pmconv2_downsample", c / 2, c, 3, 2);
    t.add("pmconv3", c / 2, 2 * c);
    t.add("pmconv4_downsample", c, 4 * c, 3, 2);
    t.add("pmconv5", 2 * c, 4 * c);
    t.add("pmconv6", 2 * c, 4 * c, 3, 1, 1, false, 1);   // ReLU gate, editline_g.py:89-90
    t.add("pmconv9", 2 * c, 4 * c);
    t.add("pmconv10", 2 * c, 4 * c);
    t.add_decoder("allconv", 4 * c, 3);
  }
  return t;
}

// ------------------------------------------------------------------------------------------ packed layers
struct ClassW {
  int ntaps = 0;
  int8_t dy[MAX_TAPS], dx[MAX_TAPS];
  float* w_direct = nullptr;   // device fp32 [tap][Ci][CoutP]
  int CoutP = 0;
  bool has_tc = false;
  C8Layer c8;                  // se_conv_c8.cu: channel-blocked input (every stride-1 layer on the bf16 path)
  bool use_c8 = false;
  // stride-2 3x3 layers on the tensor-core path read a SPACE-TO-DEPTH channel-blocked input (written that way by
  // the producing layer's epilogue): tap (ky,kx) of output (y,x) reads input row 2y+ky-1 = row y+c8dy of parity
  // (ky-1)&1, i.e. a stride-1 read at offset (c8dy, c8dx) starting at channel block c8cb = parity * Ci/8
  bool s2d = false;
  int8_t c8dy[MAX_TAPS], c8dx[MAX_TAPS], c8cb[MAX_TAPS];
  int osy = 1, ooy = 0, osx = 1, oox = 0;
  // split-half twin (SE_PREC_FP32_TC, DT_F16X2): every tap becomes three virtual taps (x_hi, w_hi), (x_hi, w_lo), (x_lo, w_hi); a
  // virtual tap reads the hi or lo channel blocks of the input (s_cb) and its weight image holds fp16(w) or fp16(w - fp16(w))
  C8Layer c8s;
  bool has_split = false;
  int s_ntaps = 0;
  float s_wscale = 1.0f;   // power of two the split-half weight images are multiplied by
  int8_t s_dy[MAX_TAPS], s_dx[MAX_TAPS], s_cb[MAX_TAPS];
};

struct Layer {
  Spec spec;
  std::string name;
  int Ci = 0;                  // stored input channels (stems are packed to 8)
  bool is_head = false;
  bool is_stem = false;
  bool set = false;
  std::vector<float> w_host, b_host;
  std::vector<ClassW> cls;
  std::vector<C8Group> groups; // deconv layers on the tensor-core path: sub-pixel classes fused per launch (se_conv_c8.h)
  int pair_cin_sum = 0;        // fused_pair: real input channels of the two source layers together (algorithmic FLOPs)
  bool fused_pair = false;     // two 5x5 stems over the same packed input fused along N (tensor-core path; see make_stem_pair)
  float* bias = nullptr;       // device [cout]
  float* w_head = nullptr;     // device [9][12][cout] (heads)
  std::vector<float> w_head_host;   // same, host copy (kernel-parameter weights of the channel-blocked head kernel)
};

}  // namespace se

using namespace se;

struct se_model {
  std::map<std::string, Layer> layers;   // key = net + "." + name
  int opt[8] = {1, 0, 0, 0, 1, 0, 0, 0};
  bool finalized = false;
  void* arena = nullptr;
  size_t arena_bytes = 0;
  std::vector<void*> owned;              // device allocations of packed weights
  // one forward at a time per model (the workspace arena is shared by every call); the model lives on ONE device; a call
  // on another stream than the previous one waits for that stream's work on the arena first
  std::mutex mu;
  // whole-forward CUDA graphs, one per call signature (entry point, shape, precision, options, every pointer argument): the
  // ~85 launches of a forward (each with its tensor-map encodes) become one cudaGraphLaunch. A signature is captured the
  // second time it is seen (one-off calls stay eager); entries die with the arena they were captured on.
  struct GraphEntry { std::vector<uintptr_t> key; cudaGraphExec_t exec = nullptr; void* arena = nullptr; int launches = 0; unsigned long long tick = 0; };
  std::vector<GraphEntry> graphs;
  std::map<std::vector<uintptr_t>, int> seen;
  unsigned long long tick = 0;
  cudaStream_t gstream = nullptr;          // graphs cannot be captured on / launched into the legacy default stream: callers that pass it
  cudaEvent_t bridge_in = nullptr, bridge_out = nullptr;   // (torch's default) are bridged through this stream with two events
  int device = -1;
  cudaStream_t last_stream = nullptr;
  bool used = false;
  cudaEvent_t order_ev = nullptr;
};

namespace se {

// 5x5 stems read an 8-channel packed input through overlapping 8-pixel windows: 64 virtual channels
// (pixel pitch 8 elements), see pack_layer / run_layer.
constexpr int STEM_PADL = 2;                       // zero pixels left of the image in the packed buffer
static inline int stem_wp(int W) { return W + 8; } // packed row length (2 left + 6 right zero pixels)
static int stored_ci(const Spec& s) { return s.k == 5 ? 64 : s.cin; }

static int upload(se_model* m, const void* host, size_t bytes, void** dev) {
  SE_CUDA_OK(cudaMalloc(dev, bytes));
  m->owned.push_back(*dev);
  SE_CUDA_OK(cudaMemcpy(*dev, host, bytes, cudaMemcpyHostToDevice));
  return 0;
}

static inline uint16_t f32_to_bf16_rn(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);
  u += 0x7fffu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}

// effective tap = sum of source taps (ky,kx) of the OIHW kernel (deconv parity classes merge taps)
// each source adds W[:, :, ky, kx] into the virtual input channels [ci_off, ci_off + cin)
struct SrcTap { int ky, kx, ci_off; };
struct EffTap { int dy, dx; std::vector<SrcTap> src; };

static int pack_class(se_model* m, Layer& L, const std::vector<EffTap>& taps, ClassW& cw) {
  const Spec& s = L.spec;
  const int Ci = L.Ci, Cout = s.cout, k = s.k;
  cw.ntaps = (int)taps.size();
  SE_REQUIRE(cw.ntaps <= MAX_TAPS, "too many taps");
  cw.CoutP = (Cout + 3) / 4 * 4;
  std::vector<float> weff((size_t)cw.ntaps * Ci * Cout, 0.0f);
  for (int t = 0; t < cw.ntaps; ++t) {
    cw.dy[t] = (int8_t)taps[t].dy;
    cw.dx[t] = (int8_t)taps[t].dx;
    for (auto& sk : taps[t].src)
      for (int ci = 0; ci < s.cin; ++ci)
        for (int co = 0; co < Cout; ++co)
          weff[((size_t)t * Ci + sk.ci_off + ci) * Cout + co] += L.w_host[(((size_t)co * s.cin + ci) * k + sk.ky) * k + sk.kx];
  }
  {
    std::vector<float> wd((size_t)cw.ntaps * Ci * cw.CoutP, 0.0f);
    for (int t = 0; t < cw.ntaps; ++t)
      for (int ci = 0; ci < Ci; ++ci)
        for (int co = 0; co < Cout; ++co) wd[((size_t)t * Ci + ci) * cw.CoutP + co] = weff[((size_t)t * Ci + ci) * Cout + co];
    int rc = upload(m, wd.data(), wd.size() * 4, (void**)&cw.w_direct);
    if (rc) return rc;
  }
  cw.has_tc = (Ci % 8 == 0) && !L.is_head;
  if (cw.has_tc) {
    cw.s2d = (s.stride == 2 && s.k == 3 && s.rate == 1 && !s.deconv && !L.is_stem && Ci % 8 == 0);
    cw.use_c8 = (s.stride == 1) || cw.s2d;
    memset(cw.c8cb, 0, sizeof(cw.c8cb));
    memcpy(cw.c8dy, cw.dy, sizeof(cw.c8dy));
    memcpy(cw.c8dx, cw.dx, sizeof(cw.c8dx));
    if (cw.s2d) {
      for (int t = 0; t < cw.ntaps; ++t) {
        const int oy = cw.dy[t], ox = cw.dx[t];          // -1, 0, +1 (input row 2y + oy)
        const int py = oy & 1, px = ox & 1;              // parity of that row / column
        cw.c8dy[t] = (int8_t)((oy - py) / 2);            // -1 for oy = -1, else 0
        cw.c8dx[t] = (int8_t)((ox - px) / 2);
        cw.c8cb[t] = (int8_t)((py * 2 + px) * (Ci / 8));
      }
    }
    SE_REQUIRE(cw.use_c8, "layer " + L.name + " has no tensor-core form");   // every gated layer of the two generators has one
    {
      int rc = c8_configure(&cw.c8, cw.ntaps, cw.c8dy, cw.c8dx, Ci, Cout, L.is_stem, cw.c8cb);
      if (rc) return rc;
    }
    TcWeights* tcp = &cw.c8.w;
    // the exact (swizzled) shared-memory image of every pipeline stage, see se_conv_tc.h. Gate channels (n >= Cout/2) are stored
    // pre-multiplied by 0.5 (exact): the accumulator then holds 0.5*g and the epilogue's sigmoid(g + b) = 0.5*tanh(0.5*g + 0.5*b) + 0.5
    // needs one add (with a constant operand) before the MUFU
    auto build_images = [&](TcWeights& tc, C8Layer* c8, const std::function<uint16_t(int, int, int)>& wv) -> int {
      const int ksteps = tc_ksteps(tc), sb = tc_stage_b_bytes(tc);
      std::vector<uint16_t> img((size_t)ksteps * sb / 2, 0);
      for (int pass = 0; pass < 2; ++pass) {
        const bool pair = pass == 1;
        if (pair && !(c8 && c8_pair_capable(*c8))) break;
        // pass 1: second copy in CTA-pair format (se_conv_c8.cu, PAIR = 1): each CTA of a pair streams only its half of the rows
        std::fill(img.begin(), img.end(), (uint16_t)0);
        for (int ks = 0; ks < ksteps; ++ks) {
          uint16_t* base = img.data() + (size_t)ks * sb / 2;
          for (int j = 0; j < tc.r64 && tc.n64; ++j) {
            const int u = ks * tc.r64 + j, t = u / tc.n64, chunk = u % tc.n64;
            for (int n = 0; n < Cout; ++n)
              for (int k = 0; k < 64; ++k) {
                const uint32_t off = pair ? c8_pair_image_offset(tc, true, j, gated_column(Cout, n), k) : tc_b_image_offset(tc.NT, tc.r64, true, j, gated_column(Cout, n), k);
                base[off / 2] = wv(t, chunk * 64 + k, n);
              }
          }
          for (int j = 0; j < tc.r32 && tc.n32; ++j) {
            const int t = ks * tc.r32 + j;
            for (int n = 0; n < Cout; ++n)
              for (int k = 0; k < 32; ++k) {
                const uint32_t off = pair ? c8_pair_image_offset(tc, false, j, gated_column(Cout, n), k)
                                          : tc_b_image_offset(tc.NT, tc.n64 ? tc.r64 : 0, false, j, gated_column(Cout, n), k);
                base[off / 2] = wv(t, tc.n64 * 64 + k, n);
              }
          }
        }
        void* d = nullptr;
        int rc = upload(m, img.data(), img.size() * 2, &d);
        if (rc) return rc;
        if (pair) c8->w_pair = d; else tc.data = d;
      }
      return 0;
    };
    auto wval = [&](int t, int ci, int n) -> float { return ci < Ci ? weff[((size_t)t * Ci + ci) * Cout + n] * (n >= Cout / 2 ? 0.5f : 1.0f) : 0.0f; };
    int rc = build_images(*tcp, cw.use_c8 ? &cw.c8 : nullptr, [&](int t, int ci, int n) -> uint16_t { return f32_to_bf16_rn(wval(t, ci, n)); });
    if (rc) return rc;
    if (cw.use_c8) {
      // ---- split-half twin: virtual tap 3t + p, p = 0: (x_hi, w_hi), 1: (x_hi, w_lo), 2: (x_lo, w_hi)
      const int CB = L.is_stem ? 1 : Ci / 8;   // channel blocks of one half of the input (the packed stem input is one block)
      cw.s_ntaps = 3 * cw.ntaps;
      SE_REQUIRE(cw.s_ntaps <= MAX_TAPS, "too many virtual taps");
      for (int t = 0; t < cw.ntaps; ++t)
        for (int pp = 0; pp < 3; ++pp) {
          cw.s_dy[3 * t + pp] = cw.c8dy[t];
          cw.s_dx[3 * t + pp] = cw.c8dx[t];
          cw.s_cb[3 * t + pp] = (int8_t)(2 * cw.c8cb[t] + (pp == 2 ? CB : 0));   // a parity group holds 2 * CB blocks
        }
      rc = c8_configure(&cw.c8s, cw.s_ntaps, cw.s_dy, cw.s_dx, Ci, Cout, L.is_stem, cw.s_cb);
      if (rc) return rc;
      // weights times a power of two (exact) that brings the largest one to [8192, 16384): the lo halves of all but negligible
      // weights are then normal fp16 numbers (22 bits for the pair); the epilogue undoes it (se_common.cuh: kSplitActScale)
      float wmax = 0.0f;
      for (int t = 0; t < cw.ntaps; ++t)
        for (int ci = 0; ci < Ci; ++ci)
          for (int n = 0; n < Cout; ++n) wmax = std::max(wmax, std::fabs(wval(t, ci, n)));
      int kw = 0;
      if (wmax > 0.0f && std::isfinite(wmax)) kw = std::min(24, std::max(0, 13 - (int)std::floor(std::log2(wmax))));
      cw.s_wscale = std::ldexp(1.0f, kw);
      auto half_bits = [](float v) -> uint16_t { return __half_as_ushort(__float2half_rn(v)); };
      rc = build_images(cw.c8s.w, &cw.c8s, [&](int vt, int ci, int n) -> uint16_t {
        const float w = wval(vt / 3, ci, n) * cw.s_wscale;
        const float hi = __half2float(__float2half_rn(w));
        return (vt % 3) == 1 ? half_bits(w - hi) : half_bits(w);
      });
      if (rc) return rc;
      cw.has_split = true;
    }
  }
  return 0;
}

static int pack_layer(se_model* m, Layer& L) {
  const Spec& s = L.spec;
  L.Ci = stored_ci(s);
  L.is_head = (s.cin == 12);
  L.is_stem = (s.k == 5);
  int rc = upload(m, L.b_host.data(), L.b_host.size() * 4, (void**)&L.bias);
  if (rc) return rc;
  if (L.is_head) {
    std::vector<float> wh((size_t)9 * 12 * s.cout);
    for (int t = 0; t < 9; ++t)
      for (int c = 0; c < 12; ++c)
        for (int o = 0; o < s.cout; ++o) wh[((size_t)t * 12 + c) * s.cout + o] = L.w_host[(((size_t)o * 12 + c) * 3 + t / 3) * 3 + t % 3];
    rc = upload(m, wh.data(), wh.size() * 4, (void**)&L.w_head);
    if (rc) return rc;
    L.w_head_host = wh;
  }
  if (L.is_stem) {
    // 5x5 / pad 2 over <= 5 real channels: K per tap would be 3-5. Instead one 64-wide GEMM-K chunk covers a
    // window of 8 horizontally adjacent pixels x 8 packed channels (kernel columns 0..4 + three zero columns):
    // 5 K-units (one per kernel row) instead of 25 taps. Window start in packed-buffer pixels:
    // (x + STEM_PADL) - 2 = x, so dx = 0.
    std::vector<EffTap> taps;
    for (int ky = 0; ky < 5; ++ky) {
      EffTap e;
      e.dy = ky - 2;
      e.dx = 0;
      for (int pxl = 0; pxl < 5; ++pxl) e.src.push_back(SrcTap{ky, pxl, pxl * 8});
      taps.push_back(e);
    }
    L.cls.resize(1);
    return pack_class(m, L, taps, L.cls[0]);
  }
  if (!s.deconv) {
    std::vector<EffTap> taps;
    const int p = s.rate * (s.k - 1) / 2;   // reference utils.py:21
    for (int ky = 0; ky < s.k; ++ky)
      for (int kx = 0; kx < s.k; ++kx) taps.push_back(EffTap{ky * s.rate - p, kx * s.rate - p, {SrcTap{ky, kx, 0}}});
    L.cls.resize(1);
    return pack_class(m, L, taps, L.cls[0]);
  }
  // nearest x2 upsample + 3x3 conv == four sub-pixel 2x2 convs over the low-res map with merged taps:
  // output row 2i   reads rows {i-1: W[0], i: W[1]+W[2]};  row 2i+1 reads {i: W[0]+W[1], i+1: W[2]}
  L.cls.resize(4);
  for (int pc = 0; pc < 4; ++pc) {
    const int py = pc / 2, px = pc % 2;
    std::vector<EffTap> taps;
    for (int a = 0; a < 2; ++a)
      for (int b = 0; b < 2; ++b) {
        EffTap e;
        e.dy = (py == 0) ? (a - 1) : a;
        e.dx = (px == 0) ? (b - 1) : b;
        std::vector<int> rows = (py == 0) ? (a == 0 ? std::vector<int>{0} : std::vector<int>{1, 2})
                                          : (a == 0 ? std::vector<int>{0, 1} : std::vector<int>{2});
        std::vector<int> cols = (px == 0) ? (b == 0 ? std::vector<int>{0} : std::vector<int>{1, 2})
                                          : (b == 0 ? std::vector<int>{0, 1} : std::vector<int>{2});
        for (int r : rows)
          for (int c : cols) e.src.push_back(SrcTap{r, c, 0});
        taps.push_back(e);
      }
    ClassW& cw = L.cls[pc];
    cw.osy = 2; cw.ooy = py; cw.osx = 2; cw.oox = px;
    rc = pack_class(m, L, taps, cw);
    if (rc) return rc;
  }
  // fuse the classes into as few launches as shared memory allows: all four (48->48), else one launch per output-row
  // parity (96->96: classes {0,1} and {2,3}); the per-class launches stay available as the fallback
  if (L.cls[0].has_tc && L.cls[0].use_c8 && L.cls[0].c8.resident && L.cls[0].c8.mode == C8_HALO) {
    for (int per : {4, 2}) {
      std::vector<C8Group> gs;
      bool ok = true;
      for (int g0 = 0; g0 < 4 && ok; g0 += per) {
        int8_t dy[C8_MAX_CLS][8], dx[C8_MAX_CLS][8];
        int ooy[C8_MAX_CLS], oox[C8_MAX_CLS];
        for (int k = 0; k < per; ++k) {
          const ClassW& cw = L.cls[g0 + k];
          for (int t = 0; t < cw.ntaps; ++t) { dy[k][t] = cw.dy[t]; dx[k][t] = cw.dx[t]; }
          ooy[k] = cw.ooy; oox[k] = cw.oox;
        }
        C8Group G;
        if (c8_configure_group(&G, per, L.cls[0].ntaps, dy, dx, ooy, oox, L.Ci, s.cout)) { ok = false; break; }
        const C8Layer& c0 = L.cls[g0].c8;
        ok = (G.geo.w.r64 == c0.w.r64 && G.geo.w.r32 == c0.w.r32 && G.geo.w.NT == c0.w.NT && G.cls_bytes == (int)tc_weight_bytes_per_image(c0.w));
        if (!ok) break;
        void* d = nullptr;
        SE_CUDA_OK(cudaMalloc(&d, (size_t)per * G.cls_bytes));
        m->owned.push_back(d);
        for (int k = 0; k < per; ++k)
          SE_CUDA_OK(cudaMemcpy((char*)d + (size_t)k * G.cls_bytes, L.cls[g0 + k].c8.w.data, G.cls_bytes, cudaMemcpyDeviceToDevice));
        G.w_all = d;
        gs.push_back(G);
      }
      if (ok) { L.groups = gs; break; }
    }
  }
  return 0;
}

// ------------------------------------------------------------------------------------------ arena
// Offsets inside one device slab, first-fit with coalescing. The forward graph is replayed twice per
// call: a dry pass (no launches) finds the peak, then the slab is grown if needed and the real pass runs.
struct Arena {
  struct Blk { size_t off, size; };
  std::vector<Blk> free_list;
  size_t top = 0, peak = 0;
  char* base = nullptr;
  void reset(char* b) { free_list.clear(); top = 0; peak = 0; base = b; }
  void* alloc(size_t bytes) {
    bytes = (bytes + 1023) & ~size_t(1023);
    for (size_t i = 0; i < free_list.size(); ++i)
      if (free_list[i].size >= bytes) {
        size_t off = free_list[i].off;
        if (free_list[i].size == bytes) free_list.erase(free_list.begin() + i);
        else { free_list[i].off += bytes; free_list[i].size -= bytes; }
        return base + off;
      }
    size_t off = top;
    top += bytes;
    if (top > peak) peak = top;
    return base + off;
  }
  void release(void* p, size_t bytes) {
    bytes = (bytes + 1023) & ~size_t(1023);
    size_t off = (char*)p - base;
    if (off + bytes == top) {
      top = off;
      // merge trailing free blocks
      bool again = true;
      while (again) {
        again = false;
        for (size_t i = 0; i < free_list.size(); ++i)
          if (free_list[i].off + free_list[i].size == top) { top = free_list[i].off; free_list.erase(free_list.begin() + i); again = true; break; }
      }
      return;
    }
    free_list.push_back({off, bytes});
    // coalesce neighbours
    bool again = true;
    while (again) {
      again = false;
      for (size_t i = 0; i < free_list.size() && !again; ++i)
        for (size_t j = 0; j < free_list.size(); ++j)
          if (i != j && free_list[i].off + free_list[i].size == free_list[j].off) {
            free_list[i].size += free_list[j].size;
            free_list.erase(free_list.begin() + j);
            again = true;
            break;
          }
    }
  }
};

struct Buf { void* p = nullptr; size_t bytes = 0; };

struct Ctx {
  se_model* m;
  cudaStream_t stream;
  int prec;
  bool dry;
  Arena arena;
  int B;
  int rc = 0;
  LaunchTag tag_;
  // label + algorithmic work of the NEXT launch (consumed by CK); see "launch timing" above
  void tag(const std::string& name, int tensor, double flops_alg, double flops_exec, double bytes_alg) {
    if (!g_timing || dry) return;
    tag_.name = name; tag_.tensor = tensor; tag_.flops_alg = flops_alg; tag_.flops_exec = flops_exec; tag_.bytes_alg = bytes_alg; tag_.set = true;
  }
  bool tc() const { return prec == SE_PREC_BF16_TC || prec == SE_PREC_FP32_TC; }   // tcgen05 kernels over channel-blocked activations
  bool split() const { return prec == SE_PREC_FP32_TC; }                            // ... in split-half storage (DT_F16X2)
  int sp() const { return split() ? 2 : 1; }                                        // channel-block multiplier of that storage
  int act_dt() const { return prec == SE_PREC_FP32_EXACT ? DT_F32 : (split() ? DT_F16X2 : DT_BF16); }
  size_t esz() const { return (prec == SE_PREC_FP32_EXACT || split()) ? 4 : 2; }
  Buf get(size_t bytes) { Buf b; b.bytes = bytes; b.p = arena.alloc(bytes); return b; }
  void put(Buf& b) { if (b.p) arena.release(b.p, b.bytes); b.p = nullptr; }
};

#define CK(expr)                                                    \
  do {                                                              \
    if (!c.dry) {                                                   \
      size_t _slot = 0;                                             \
      const bool _timed = g_timing;                                 \
      if (_timed) { int _rt = timing_begin(c.tag_, c.stream, &_slot); if (_rt) { c.rc = _rt; return _rt; } } \
      c.tag_.set = false;                                           \
      int _rc = (expr);                                             \
      if (_rc) { c.rc = _rc; return _rc; }                          \
      if (_timed) { int _rt = timing_end(_slot, c.stream); if (_rt) { c.rc = _rt; return _rt; } } \
      ++g_launches;                                                 \
    }                                                               \
  } while (0)

// activation view. c8 == 0: NHWC, channels [0,C) at pixel pitch ld. c8 == 1: [B][ld blocks][H][W][8], the view's
// channels start at block cb_off.
struct View { void* p; int H, W, C, ld; int c8 = 0; int cb_off = 0; };
static inline View nhwc(void* p, int H, int W, int C, int ld) { View v; v.p = p; v.H = H; v.W = W; v.C = C; v.ld = ld; return v; }
static inline View c8view(void* p, int H, int W, int C, int cbtot, int cb_off) { View v; v.p = p; v.H = H; v.W = W; v.C = C; v.ld = cbtot; v.c8 = 1; v.cb_off = cb_off; return v; }
static inline size_t act_bytes(const struct Ctx& c, int H, int W, int C, int c8);

static Layer* find_layer(se_model* m, char net, const std::string& name) {
  auto it = m->layers.find(std::string(1, net) + "." + name);
  return it == m->layers.end() ? nullptr : &it->second;
}
// layer that has weights (forward paths); nullptr + error text otherwise
static Layer* find_ready(se_model* m, char net, const std::string& name) {
  Layer* L = find_layer(m, net, name);
  if (L && !L->set) {
    set_error(std::string("weights of net") + net + " were never loaded (layer " + name + ")");
    return nullptr;
  }
  return L;
}

static int launch_conv(Ctx& c, const ConvParams& cp, const ClassW& cw) {
  if (c.split() && cw.has_split) return c8_launch(cp, cw.c8s, c.stream);
  if (c.prec == SE_PREC_BF16_TC && cw.has_tc) return c8_launch(cp, cw.c8, c.stream);
  ConvParams d = cp;
  d.w = cw.w_direct;
  return direct_launch(d, cw.CoutP, c.prec == SE_PREC_FP32_EXACT, c.stream);
}

// one gated conv / deconv layer: in (Hi x Wi x Ci) -> out view (channels written at [choff, choff+cout_g))
// layout a layer wants for its input on the bf16 tensor-core path (stride-2 layers read NHWC, the rest C8)
// 0 NHWC, 1 channel-blocked (C8), 2 channel-blocked space-to-depth (stride-2 layers)
static int wants_c8(const Ctx& c, const Layer& L) {
  if (!c.tc() || L.is_head) return 0;
  if (L.spec.stride == 1) return 1;
  return (!L.cls.empty() && L.cls[0].s2d) ? 2 : 0;
}
static inline size_t act_bytes(const Ctx& c, int H, int W, int C, int c8) {
  return c8 ? (size_t)c.B * ((C + 7) / 8) * H * W * 16 * c.sp() : (size_t)c.B * H * W * C * c.esz();
}
// the packed 8-channel network input (zero-padded rows of stem_wp(W) pixels): NHWC with C = ld = 8 for the CUDA-core
// kernels, the same bytes seen as one channel block of width stem_wp(W) for the tensor-core path
static View stem_view(const Ctx& c, void* p, int H, int W) {
  if (c.tc()) return c8view(p, H, W, 8, c.sp(), 0);
  return nhwc(p, H, W, 8, 8);
}

static int run_layer(Ctx& c, Layer& L, const View& in, void* out, int ldo, int choff, int out_c8 = 0) {
  SE_REQUIRE(in.c8 == wants_c8(c, L), "activation layout mismatch at layer " + L.name);
  const Spec& s = L.spec;
  const int Ho = s.deconv ? in.H : (in.H + s.stride - 1) / s.stride;   // position grid
  const int Wo = s.deconv ? in.W : (in.W + s.stride - 1) / s.stride;
  const bool fused = c.prec == SE_PREC_BF16_TC && !L.groups.empty() && in.c8 == 1;
  const bool split = c.split();
  const int n_launch = fused ? (int)L.groups.size() : (int)L.cls.size();
  for (int li = 0; li < n_launch; ++li) {
    const C8Group* grp = fused ? &L.groups[li] : nullptr;
    ClassW& cw = L.cls[fused ? li * grp->ncls : li];
    ConvParams cp;
    memset(&cp, 0, sizeof(cp));
    cp.x = in.p; cp.in_dt = c.act_dt();
    cp.N = c.B; cp.Hi = in.H; cp.Wi = in.W; cp.Ci = L.Ci; cp.ldx = in.ld;
    if (L.is_stem && !in.c8) {   // `in` is the packed 8-channel buffer with zero-padded rows of stem_wp(W) pixels
      cp.ldx = 8;
      cp.Wi = stem_wp(in.W) - 7;
      cp.x_row_pitch = (long long)stem_wp(in.W) * 8;
      cp.x_img_pitch = (long long)in.H * cp.x_row_pitch;
    }
    if (in.c8) {
      cp.in_c8 = 1; cp.x_cb_off = in.cb_off; cp.ldx = in.ld;
      if (L.is_stem) cp.Wi = stem_wp(in.W);   // the window starts at buffer pixel x (image sits at x + STEM_PADL)
    }
    cp.out_c8 = out_c8;
    cp.Ho = Ho; cp.Wo = Wo; cp.stride = s.deconv ? 1 : s.stride;
    cp.ntaps = cw.ntaps;
    memcpy(cp.dy, cw.dy, sizeof(cp.dy));
    memcpy(cp.dx, cw.dx, sizeof(cp.dx));
    if (split) {
      SE_REQUIRE(cw.has_split && in.c8 && out_c8, "split-half mode runs on channel-blocked activations (layer " + L.name + ")");
      cp.f16x2 = 1;
      // hi blocks first, lo blocks after them: per image (channel-blocked) or per parity group (space-to-depth)
      cp.out_split_stride = out_c8 == 2 ? (long long)(ldo / 8) * (Ho * cw.osy / 2) * (Wo * cw.osx / 2) : (long long)(ldo / 2) * (Ho * cw.osy) * (Wo * cw.osx);
    }
    if (in.c8 == 2) {   // space-to-depth input: a stride-1 problem on the half-resolution grid with per-tap parity blocks
      SE_REQUIRE(cw.s2d && in.H % 2 == 0 && in.W % 2 == 0, "space-to-depth input at layer " + L.name);
      cp.Hi = in.H / 2; cp.Wi = in.W / 2; cp.stride = 1;
      memcpy(cp.dy, cw.c8dy, sizeof(cp.dy));
      memcpy(cp.dx, cw.c8dx, sizeof(cp.dx));
      memcpy(cp.tap_cb, cw.c8cb, sizeof(cp.tap_cb));
    }
    if (split) {        // the virtual taps of the split-half twin (already in space-to-depth form where that applies)
      cp.ntaps = cw.s_ntaps;
      memcpy(cp.dy, cw.s_dy, sizeof(cp.dy));
      memcpy(cp.dx, cw.s_dx, sizeof(cp.dx));
      memcpy(cp.tap_cb, cw.s_cb, sizeof(cp.tap_cb));
    }
    cp.w = nullptr; cp.w_img_stride = 0;
    cp.bias = L.bias; cp.bias_host = L.b_host.data(); cp.Cout = s.cout;
    cp.y = out; cp.out_dt = c.act_dt();
    cp.Hout = Ho * cw.osy; cp.Wout = Wo * cw.osx; cp.ldo = ldo; cp.choff = choff;
    cp.osy = cw.osy; cp.ooy = cw.ooy; cp.osx = cw.osx; cp.oox = cw.oox;
    cp.epi = s.act == 1 ? EPI_GATE_RELU : EPI_GATE_ELU;
    cp.scale = split ? 1.0f / (kSplitActScale * cw.s_wscale) : 1.0f;   // split-half: accumulator -> true pre-activation (exact: powers of two)
    cp.colscale = nullptr;
    if (L.fused_pair) {
      // two space-to-depth tensors of 4 x 3 blocks each, back to back per image (ldo = 24 blocks): blocks 3..5 of the fused
      // output are blocks 0..2 of the second one, 12 - 3 = 9 block planes further on
      SE_REQUIRE(out_c8 == 2 && ldo == 24, "a fused stem pair writes two space-to-depth tensors");
      cp.out_blk_split = 3; cp.out_par_stride = 3; cp.out_blk_jump = 9 * (cp.Hout / 2) * (cp.Wout / 2);
    }
    if (g_timing && !c.dry) {
      // algorithmic work of this launch. A deconv layer is 4 sub-pixel class launches: each gets a quarter of the
      // reference op's 2*MAC (nearest x2 + 3x3 over the (2Ho x 2Wo) output) and issues 4 taps instead of 9.
      // (a fused launch carries `gc` classes)
      const double gc = grp ? grp->ncls : 1.0;
      const double pos = (double)c.B * Ho * Wo * gc, ncls = (double)L.cls.size() / gc;
      const double cin_alg = L.fused_pair ? L.pair_cin_sum / 2.0 : (double)s.cin;   // a stem pair: two 48-output layers over their own channels
      const double f_alg = 2.0 * pos * s.cout * cin_alg * (s.deconv ? 9.0 : (double)s.k * s.k);
      const double f_exec = 2.0 * pos * s.cout * cin_alg * (s.deconv ? 4.0 : (double)s.k * s.k) * (split ? 3.0 : 1.0);   // split-half: 3 products per tap
      const double bytes = ((double)c.B * in.H * in.W * (L.fused_pair ? 8.0 : (double)s.cin) / ncls + pos * (s.cout / 2) + (double)s.cout * s.cin * s.k * s.k / ncls) * c.esz();
      const bool tcp = c.tc() && cw.has_tc;
      char buf[160];
      snprintf(buf, sizeof(buf), "%s|%s %d->%d k%d s%d d%d @%dx%d", tcp ? (split ? "conv_c8_kernel (split-half fp16 x3)" : "conv_c8_kernel") : "conv_direct_kernel",
               s.deconv ? (grp ? (grp->ncls == 4 ? "deconv (4 classes fused)" : "deconv (2 classes fused)") : "deconv-class") : (L.fused_pair ? "stem pair" : "conv"), s.cin, s.cout, s.k, s.stride, s.rate, Ho * cw.osy, Wo * cw.osx);
      c.tag(buf, tcp ? 1 : 0, f_alg, f_exec, bytes);
    }
    if (grp) CK(c8_launch(cp, cw.c8, c.stream, grp));
    else CK(launch_conv(c, cp, cw));
  }
  static const bool dbg = getenv("SE_DEBUG_NAN") != nullptr;
  if (dbg && !c.dry && c.act_dt() == DT_BF16 && !split) {
    const int cg = s.cout / 2, Hout = Ho * L.cls[0].osy, Wout = Wo * L.cls[0].osx;
    const long long n_out = out_c8 ? (long long)c.B * ldo * Hout * Wout * 8 : (long long)c.B * Hout * Wout * ldo;
    const long long n_in = in.c8 ? (long long)c.B * in.ld * in.H * (L.is_stem ? stem_wp(in.W) : in.W) * 8 / (in.c8 == 2 ? 4 : 1) : (long long)c.B * in.H * in.W * in.ld;
    fprintf(stderr, "[nan] %-28s in %dx%d c8=%d ld=%d nonfinite_in=%lld | out %dx%d c8=%d ld=%d choff=%d cg=%d nonfinite_out(buffer)=%lld use_c8=%d mode=%d res=%d\n", L.name.c_str(), in.H, in.W,
            in.c8, in.ld, count_nonfinite_bf16(in.p, n_in, c.stream), Hout, Wout, out_c8, ldo, choff, cg, count_nonfinite_bf16(out, n_out, c.stream), (int)L.cls[0].use_c8,
            L.cls[0].c8.mode, (int)L.cls[0].c8.resident);
  }
  return 0;
}

static void out_dims(const Spec& s, int H, int W, int* Ho, int* Wo) {
  if (s.deconv) { *Ho = 2 * H; *Wo = 2 * W; }
  else { *Ho = (H + s.stride - 1) / s.stride; *Wo = (W + s.stride - 1) / s.stride; }
}

// run a chain of gated layers; intermediate buffers come from the arena. Each intermediate is written in the layout
// its consumer wants. The last layer writes to (final_out, final_ld, final_choff, final_c8) when given, else to a
// fresh buffer (layout final_c8) returned in *res.
static int run_chain(Ctx& c, char net, const std::vector<std::string>& names, View in, bool free_in, Buf in_buf, View* res, Buf* res_buf,
                     void* final_out = nullptr, int final_ld = 0, int final_choff = 0, int final_c8 = -1) {
  View cur = in;
  Buf cur_buf = in_buf;
  bool cur_owned = free_in;
  if (final_c8 < 0) final_c8 = c.tc() ? 1 : 0;
  for (size_t i = 0; i < names.size(); ++i) {
    Layer* L = find_ready(c.m, net, names[i]);
    SE_REQUIRE(L != nullptr, "unknown or unloaded layer " + names[i] + ": " + last_error());
    int Ho, Wo;
    out_dims(L->spec, cur.H, cur.W, &Ho, &Wo);
    const int cg = L->spec.cout / 2;
    const bool last = (i + 1 == names.size());
    View nxt;
    Buf nb;
    if (last && final_out) {
      nxt = final_c8 ? c8view(final_out, Ho, Wo, cg, final_ld, final_choff / 8) : nhwc(final_out, Ho, Wo, cg, final_ld);
      int rc = run_layer(c, *L, cur, final_out, final_ld, final_choff, final_c8);
      if (rc) return rc;
    } else {
      int oc8 = final_c8;
      if (!last) {
        Layer* nx = find_ready(c.m, net, names[i + 1]);
        SE_REQUIRE(nx != nullptr, "unknown or unloaded layer " + names[i + 1]);
        oc8 = wants_c8(c, *nx);
      }
      nb = c.get(act_bytes(c, Ho, Wo, cg, oc8));
      nxt = oc8 ? c8view(nb.p, Ho, Wo, cg, (cg + 7) / 8 * c.sp(), 0) : nhwc(nb.p, Ho, Wo, cg, cg);
      if (oc8 == 2) { nxt.c8 = 2; nxt.ld = 4 * (cg / 8) * c.sp(); }   // [N][4*cg/8][Ho/2][Wo/2][8] (split-half: twice the blocks per parity)
      int rc = run_layer(c, *L, cur, nb.p, oc8 ? nxt.ld : cg, 0, oc8);
      if (rc) return rc;
    }
    if (cur_owned) c.put(cur_buf);
    cur = nxt;
    cur_buf = nb;
    cur_owned = !(last && final_out);
  }
  if (res) *res = cur;
  if (res_buf) *res_buf = cur_buf;
  return 0;
}

static std::vector<std::string> with_prefix(const std::string& pfx, std::initializer_list<const char*> l) {
  std::vector<std::string> v;
  for (auto s : l) v.push_back(pfx + s);
  return v;
}

// out_bs / msoft_bs: elements between images of out_nchw / mask_soft (0 = dense); non-zero when they are views into a packed
// [B,4,H,W] output (se_forward_inference_packed)
static int run_head(Ctx& c, char net, const std::string& name, const View& in, int mode, const float* img, const float* mask_bin,
                    const float* mask_soft, float* out_nchw, float* out2, void* out_pack8, long long out_bs = 0, long long msoft_bs = 0,
                    unsigned char* out_u8 = nullptr) {
  Layer* L = find_ready(c.m, net, name);
  SE_REQUIRE(L != nullptr && L->is_head, "head layer " + name + ": " + last_error());
  {
    // 12-channel map in (two channel blocks on the C8 path), image / mask planes in, cout (+ blend / pack) planes out
    const double px = (double)c.B * in.H * in.W;
    const double bytes = px * ((in.c8 ? 16 : 12) * c.esz() + (img ? 12 : 0) + (mask_bin ? 4 : 0) + (mask_soft ? 4 : 0) + (out_nchw ? 4 * L->spec.cout : 0) +
                               (out2 ? 4 * (mode == HEAD_MASK ? 1 : L->spec.cout) : 0) + (out_pack8 ? 8 * c.esz() : 0));
    const double fl = 2.0 * px * 9 * 12 * L->spec.cout;
    c.tag(std::string(in.c8 == 1 && c.act_dt() == DT_BF16 ? "head_c8_kernel" : "head_kernel") + "|12->" + std::to_string(L->spec.cout) + " k3 + " +
              (mode == HEAD_MASK ? "sigmoid+threshold" : mode == HEAD_TANH ? "tanh" : mode == HEAD_COARSE ? "tanh+blend+pack8" : "tanh+soft blend"),
          0, fl, fl, bytes);
  }
  if (c.split()) {
    SE_REQUIRE(in.c8 == 1 && in.ld == 4, "split-half head input: two channel blocks, hi + lo");
    CK(head_split(in.p, L->w_head, L->bias, L->spec.cout, c.B, in.H, in.W, mode, img, mask_bin, mask_soft, out_nchw, out2, out_pack8,
                  c.m->opt[SE_OPT_NO_MASK_COARSE], stem_wp(in.W), STEM_PADL, out_bs, msoft_bs, out_u8, c.stream));
    return 0;
  }
  if (in.c8 == 1 && c.act_dt() == DT_BF16) {
    CK(head_c8(in.p, L->w_head_host.data(), L->b_host.data(), L->spec.cout, c.B, in.H, in.W, mode, img, mask_bin, mask_soft, out_nchw, out2,
               out_pack8, c.m->opt[SE_OPT_NO_MASK_COARSE], stem_wp(in.W), STEM_PADL, out_bs, msoft_bs, out_u8, c.stream));
    return 0;
  }
  CK(head(in.p, c.act_dt(), in.c8, L->w_head, L->bias, L->spec.cout, c.B, in.H, in.W, mode, img, mask_bin, mask_soft, out_nchw, out2,
          out_pack8, c.m->opt[SE_OPT_NO_MASK_COARSE], stem_wp(in.W), STEM_PADL, out_bs, msoft_bs, out_u8, c.stream));
  return 0;
}

// ------------------------------------------------------------------------------------------ contextual attention
// cam_1 + cam_2 (reference splitcam.py:57-108,147-174) on an NHWC feature map f [B,h,w,C]:
//   S = Q K^T  as a stride-2, 4x4-tap "convolution" of f with per-image kernels K   (utils.py:72-99)
//   A = softmax_l(10 * S * m_l),  out = fold_sum(A V) as four sub-pixel 2x2 convolutions over A
// bf16 tensor-core path (se_cam.cu): f is the space-to-depth channel-blocked map, out is channel-blocked [B][12][h][w][8]
static int run_cam_tc(Ctx& c, const View& f, const float* mask_s, void* out, float* attn_out) {
  SE_REQUIRE(f.c8 == 2 && f.C == 96, "tensor-core attention reads a 96-channel space-to-depth channel-blocked map");
  CamPlan pl;
  int rc = cam_plan(c.B, f.H, f.W, &pl);
  if (rc) return rc;
  Buf fn = c.get(pl.fn_bytes), cs = c.get(pl.cs_bytes), P = c.get(pl.p_bytes);
  if (g_timing && !c.dry) {
    const double L = (double)pl.hs * pl.ws;
    const double fl = 4.0 * c.B * L * L * 96 * 16;   // QK^T + PV (SURVEY.md 8d); the statistics sweep repeats QK^T: executed = 1.5x
    c.tag("cam_s_kernel + cam_pv_kernel (+ norm, colscale)|contextual attention", 1, fl, 1.5 * fl,
          (double)c.B * f.H * f.W * 96 * 2 * 2 + 2.0 * (double)pl.p_bytes);
  }
  CK(cam_forward_tc(f.p, mask_s, out, pl, fn.p, (float*)cs.p, P.p, attn_out, c.stream));
  if (!c.dry) g_launches += 3;   // four kernels behind one call
  c.put(P); c.put(cs); c.put(fn);
  return 0;
}

static int run_cam(Ctx& c, const View& f, const float* mask_s, void* out, int out_ld, float* attn_out /*fp32 [B,L,N] or null*/, int out_c8 = 0) {
  SE_REQUIRE(f.c8 == 0, "attention reads an NHWC feature map");
  const int B = c.B, h = f.H, w = f.W, C = f.C;
  SE_REQUIRE(h % 2 == 0 && w % 2 == 0 && h >= 4 && w >= 4, "attention map must be even-sized and >= 4");
  const int hs = (h - 4) / 2 + 1, ws = (w - 4) / 2 + 1, L = hs * ws;
  const int Lpad = (L + 127) / 128 * 128;
  // CUDA-core path (fp32 modes, the bf16 cross-check, and channel counts other than netG's 96): the tensor-core attention is
  // run_cam_tc / se_cam.cu
  const int dt = c.act_dt();

  Buf rnorm = c.get((size_t)B * C * 4);
  Buf colm = c.get((size_t)B * L * 4);
  c.tag("plane_sumsq/rnorm|attention key norm", 0, 0, 0, (double)B * h * w * C * c.esz());
  CK(plane_reduce(f.p, dt, B, h * w, C, f.ld, 0, RED_RNORM, (float*)rnorm.p, c.stream));
  c.tag("cam_colmask_kernel", 0, 0, 0, (double)B * h * w * 4);
  CK(cam_colmask(mask_s, (float*)colm.p, B, h, w, hs, ws, 0.1f, c.stream));

  // ---- keys
  const size_t kbytes = (size_t)B * 16 * C * Lpad * 4;   // keys as per-image conv kernels: fp32 [b][tap][c][Lpad]
  Buf kbuf = c.get(kbytes);
  SE_REQUIRE(f.ld == C, "attention input must be dense NHWC");
  c.tag("cam_pack_k|attention key operand", 0, 0, 0, (double)B * h * w * C * c.esz() + (double)kbytes);
  CK(cam_pack_k(f.p, dt, (const float*)rnorm.p, kbuf.p, B, h, w, C, ws, L, Lpad, c.stream));

  // ---- logits S[b, n, l] (fp32, row pitch Lpad), scaled by 10 * m_l in the GEMM epilogue
  Buf sbuf = c.get((size_t)B * L * Lpad * 4);
  {
    ConvParams cp;
    memset(&cp, 0, sizeof(cp));
    cp.x = f.p; cp.in_dt = dt; cp.N = B; cp.Hi = h; cp.Wi = w; cp.Ci = C; cp.ldx = f.ld;
    cp.Ho = hs; cp.Wo = ws; cp.stride = 2; cp.ntaps = 16;
    for (int t = 0; t < 16; ++t) { cp.dy[t] = (int8_t)(t / 4); cp.dx[t] = (int8_t)(t % 4); }
    cp.bias = nullptr; cp.Cout = L;
    cp.y = sbuf.p; cp.out_dt = DT_F32; cp.Hout = hs; cp.Wout = ws; cp.ldo = Lpad; cp.choff = 0;
    cp.osy = 1; cp.ooy = 0; cp.osx = 1; cp.oox = 0;
    cp.epi = EPI_LINEAR; cp.scale = 10.0f; cp.colscale = (const float*)colm.p;
    ClassW cw;
    cw.ntaps = 16;
    cw.CoutP = Lpad;
    cw.w_direct = (float*)kbuf.p;
    cp.w_img_stride = (long long)16 * C * Lpad;
    c.tag("conv_direct_kernel|attention S=QK^T", 0, 2.0 * B * L * (double)L * C * 16,
          2.0 * B * L * (double)L * C * 16, (double)B * h * w * C * c.esz() + (double)kbytes + (double)B * L * Lpad * 4);
    CK(launch_conv(c, cp, cw));
  }
  c.put(kbuf);
  c.put(rnorm);

  // ---- softmax over keys -> P[b, n, 0..Lpad)
  Buf pbuf = c.get((size_t)B * L * Lpad * c.esz());
  c.tag("softmax_rows|attention", 0, 0, 0, (double)B * L * Lpad * (4 + c.esz()));
  CK(softmax_rows((const float*)sbuf.p, Lpad, pbuf.p, dt, Lpad, (long long)B * L, L, c.stream));
  if (attn_out) {
    // cam_1 returns [B, L(keys), hs, ws]: transpose of P
    // (small, test-only path: done with the generic layout kernel, P viewed as NHWC with C = L keys)
    if (dt == DT_F32) CK(nhwc_to_nchw(pbuf.p, dt, attn_out, B, L, L, Lpad, 0, c.stream));
    else CK(nhwc_to_nchw(pbuf.p, dt, attn_out, B, L, L, Lpad, 0, c.stream));
  }
  c.put(sbuf);
  c.put(colm);

  // ---- values + fold-sum
  const size_t per_pc_bytes = (size_t)B * 4 * Lpad * C * 4;   // values per sub-pixel class: fp32 [b][tap][key][c]
  Buf vbuf = c.get(4 * per_pc_bytes);
  c.tag("cam_pack_v|attention value operand", 0, 0, 0, (double)B * h * w * C * c.esz() + 4.0 * per_pc_bytes);
  CK(cam_pack_v(f.p, dt, vbuf.p, B, h, w, C, ws, L, Lpad, c.stream));
  for (int pc = 0; pc < 4; ++pc) {
    ConvParams cp;
    memset(&cp, 0, sizeof(cp));
    cp.x = pbuf.p; cp.in_dt = dt; cp.N = B; cp.Hi = hs; cp.Wi = ws; cp.Ci = Lpad; cp.ldx = Lpad;
    cp.Ho = h / 2; cp.Wo = w / 2; cp.stride = 1; cp.ntaps = 4;
    for (int t = 0; t < 4; ++t) { cp.dy[t] = (int8_t)(-(t / 2)); cp.dx[t] = (int8_t)(-(t % 2)); }
    cp.bias = nullptr; cp.Cout = C;
    cp.y = out; cp.out_dt = dt; cp.Hout = h; cp.Wout = w; cp.ldo = out_c8 ? (C + 7) / 8 : out_ld; cp.choff = 0;
    cp.out_c8 = out_c8;
    cp.osy = 2; cp.ooy = pc / 2; cp.osx = 2; cp.oox = pc % 2;
    cp.epi = EPI_LINEAR; cp.scale = 1.0f; cp.colscale = nullptr;
    ClassW cw;
    cw.ntaps = 4;
    cw.CoutP = C;
    cw.w_direct = reinterpret_cast<float*>((char*)vbuf.p + pc * per_pc_bytes);
    cp.w_img_stride = (long long)4 * Lpad * C;
    c.tag("conv_direct_kernel|attention out=fold(PV) class", 0,
          2.0 * B * (h / 2) * (w / 2) * (double)C * L * 4, 2.0 * B * (h / 2) * (w / 2) * (double)C * L * 4,
          ((double)B * L * Lpad + (double)B * 4 * Lpad * C + (double)B * (h / 2) * (w / 2) * C) * c.esz());
    CK(launch_conv(c, cp, cw));
  }
  c.put(vbuf);
  c.put(pbuf);
  return 0;
}

// Attention of the fp32-on-tensor-cores mode: f fp32 NHWC [B][h][w][96] -> out fp32 NHWC, split-half fp16 tcgen05 GEMMs (se_gemm_split.cu)
static int run_cam_split(Ctx& c, const float* f, int h, int w, int C, const float* mask_s, float* out) {
  CamSplitPlan pl;
  {
    int rc = cam_split_plan(c.B, h, w, C, &pl);
    if (rc) return rc;
  }
  Buf rnorm = c.get((size_t)c.B * C * 4), colm = c.get((size_t)c.B * pl.L * 4);
  Buf q = c.get(pl.q_bytes), kn = c.get(pl.q_bytes), sb = c.get(pl.s_bytes), pb = c.get(pl.p_bytes), ob = c.get(pl.o_bytes);
  c.tag("plane_sumsq/rnorm|attention key norm", 0, 0, 0, (double)c.B * h * w * C * 4);
  CK(plane_reduce(f, DT_F32, c.B, h * w, C, C, 0, RED_RNORM, (float*)rnorm.p, c.stream));
  c.tag("cam_colmask_kernel", 0, 0, 0, (double)c.B * h * w * 4);
  CK(cam_colmask(mask_s, (float*)colm.p, c.B, h, w, pl.hs, pl.ws, 0.1f, c.stream));
  const double fl = 2.0 * c.B * (double)pl.L * pl.L * pl.KQ * 2.0;   // S and PV, algorithmic (one product each)
  c.tag("gemm_split_kernel x2 (split-half fp16 x3) + pack / softmax / fold|contextual attention", 1, fl, 3.0 * 2.0 * c.B * (double)pl.Mp * pl.Mp * pl.KQ * 2.0,
        (double)c.B * h * w * C * 4 * 2 + 2.0 * pl.q_bytes * 2 + 2.0 * pl.s_bytes + 2.0 * pl.p_bytes + 2.0 * pl.o_bytes);
  CK(cam_forward_split(f, (const float*)rnorm.p, (const float*)colm.p, out, pl, q.p, kn.p, (float*)sb.p, pb.p, (float*)ob.p, c.stream));
  if (!c.dry) g_launches += 4;   // pack, S GEMM, softmax, PV GEMM, fold behind one call
  c.put(ob); c.put(pb); c.put(sb); c.put(kn); c.put(q); c.put(colm); c.put(rnorm);
  return 0;
}

// ------------------------------------------------------------------------------------------ networks
static const std::initializer_list<const char*> kTrunk9 = {"conv1", "conv2_downsample", "conv3", "conv4_downsample", "conv5",
                                                           "conv6", "conv7_atrous", "conv8_atrous", "conv9_atrous"};

// input packing / pooling glue in the activation storage of the current mode
static int do_pack8(Ctx& c, const float* img, const float* sk, const float* mask, void* out, int H, int W, int img_mode, float sscale, int write_mask,
                    int img2_mode = -1) {
  if (c.split()) return pack8_split(img, sk, mask, out, c.B, H, W, stem_wp(W), STEM_PADL, img_mode, sscale, write_mask, c.stream);
  return pack8(img, sk, mask, out, c.act_dt(), c.B, H, W, stem_wp(W), STEM_PADL, img_mode, sscale, write_mask, c.stream, img2_mode);
}
static int do_pool_broadcast(Ctx& c, const View& v, int HW, int mode, float* pooled, void* cat, int cat_ld, int tc) {
  if (c.split()) {
    int rc = plane_reduce_split(v.p, c.B, HW, 96, v.ld / 2, mode, pooled, c.stream);
    if (rc) return rc;
    return broadcast_split(pooled, cat, c.B, HW, 96, cat_ld / 2, 96, c.stream);
  }
  int rc = plane_reduce(v.p, c.act_dt(), c.B, HW, 96, v.ld, v.c8, mode, pooled, c.stream);
  if (rc) return rc;
  return broadcast_channels(pooled, cat, c.act_dt(), c.B, HW, 96, cat_ld, 96, tc, c.stream);
}

// MDGenerator.forward: x [B,3,H,W], guide [B,1,H,W] -> mask1 (soft, NCHW), optional x_stage1; also the
// binarised mask plane (mask1 > 0.5) when mask_bin != nullptr.
static int run_netM(Ctx& c, const float* x, const float* guide, int H, int W, float* mask1, float* x_stage1, float* mask_bin, long long mask1_bs = 0,
                    unsigned char* mask_u8 = nullptr) {
  const int dt = c.act_dt();
  Buf in8 = c.get((size_t)c.B * H * stem_wp(W) * 8 * c.esz());
  c.tag("pack8_kernel|mask-mul + concat + cast", 0, 0, 0, (double)c.B * H * W * 20 + (double)c.B * H * stem_wp(W) * 8 * c.esz());
  CK(do_pack8(c, x, guide, nullptr, in8.p, H, W, PACK_IMG_ONE, 1.0f, 0));
  View x9;
  Buf b9;
  int rc = run_chain(c, 'M', with_prefix("", kTrunk9), stem_view(c, in8.p, H, W), true, in8, &x9, &b9);
  if (rc) return rc;
  if (x_stage1) {
    // image decoder consumes the conv9 output (editline2_g.py:76-77)
    View v16;
    Buf b16;
    rc = run_chain(c, 'M', with_prefix("conv", {"11", "12", "13_upsample_conv", "14", "15_upsample_conv", "16"}), x9, false, Buf(), &v16, &b16);
    if (rc) return rc;
    rc = run_head(c, 'M', "conv17", v16, HEAD_TANH, nullptr, nullptr, nullptr, x_stage1, nullptr, nullptr);
    if (rc) return rc;
    c.put(b16);
  }
  View v;
  Buf b;
  rc = run_chain(c, 'M', with_prefix("", {"conv10_atrous", "conv_mask_11", "conv_mask_12", "conv_mask_13_upsample_conv", "conv_mask_14",
                                          "conv_mask_15_upsample_conv", "conv_mask_16"}),
                 x9, true, b9, &v, &b);
  if (rc) return rc;
  Buf scratch;
  float* mb = mask_bin;
  if (!mb) { scratch = c.get((size_t)c.B * H * W * 4); mb = (float*)scratch.p; }
  rc = run_head(c, 'M', "conv_mask_17", v, HEAD_MASK, nullptr, nullptr, nullptr, mask1, mb, nullptr, mask1_bs, 0, mask_u8);
  if (rc) return rc;
  c.put(scratch);
  c.put(b);
  return 0;
}

// DeepFillC2Generator.forward. x, x2 [B,3,H,W]; mask, mask2 planes [B,H,W]; guide [B,H,W] or null (ones).
// Outputs: x_stage1 (optional), x_stage2 (optional NCHW), composed (optional: fine*soft + img*(1-soft)).
static int run_netG(Ctx& c, const float* x, const float* x2, const float* mask, const float* mask2, const float* guide, int H, int W,
                    float* x_stage1, float* x_stage2, float* composed, const float* mask_soft, const float* blend_img,
                    long long composed_bs = 0, long long msoft_bs = 0, unsigned char* composed_u8 = nullptr) {
  // guide == nullptr: the reference's guide=None -> an all-ones sketch channel (editline_g.py:127-130), built by pack8
  const int dt = c.act_dt();
  const int* opt = c.m->opt;
  const int h = H / 4, w = W / 4;
  const size_t e = c.esz();

  // ---- stage 1: coarse encoder + style ("warp-in") encoder -> 192-channel concat -> coarse decoder
  const int tc = c.tc() ? 1 : 0;
  const int cat_ld = tc ? 24 * c.sp() : 192;           // 192-channel concat buffers: 24 channel blocks (x2 split-half) or pixel pitch 192
  auto cat_view = [&](void* p) { return tc ? c8view(p, h, w, 192, cat_ld, 0) : nhwc(p, h, w, 192, 192); };
  Buf cat1 = c.get((size_t)c.B * h * w * 192 * e);
  // stem pairs (tensor-core path, make_stem_pair): conv1 + wconv1 share one packed input when both encoders see the same image
  // and mask (always true on the inference path: netG(inputs, inputs, mask_bin, mask_bin, line))
  Layer* pair1 = (c.prec == SE_PREC_BF16_TC && x == x2 && mask == mask2) ? find_layer(c.m, 'G', "conv1+wconv1") : nullptr;
  Layer* pair2 = c.prec == SE_PREC_BF16_TC ? find_layer(c.m, 'G', "xconv1+pmconv1") : nullptr;
  const size_t pair_bytes = (size_t)c.B * 24 * (H / 2) * (W / 2) * 16;   // two space-to-depth tensors of 24 channels
  auto pair_view = [&](void* p, int which) { View v = c8view(p, H, W, 24, 24, 12 * which); v.c8 = 2; return v; };
  std::vector<std::string> trunk_rest(kTrunk9.begin() + 1, kTrunk9.end());   // conv2_downsample .. conv9_atrous
  if (pair1) {
    Buf in8 = c.get((size_t)c.B * H * stem_wp(W) * 8 * e);
    c.tag("pack8_kernel|mask-mul + concat + cast", 0, 0, 0, (double)c.B * H * W * 20 + (double)c.B * H * stem_wp(W) * 8 * c.esz());
    CK(do_pack8(c, x, guide, mask, in8.p, H, W, PACK_IMG_ONE_MINUS_M, 1.0f, 1, opt[SE_OPT_NO_MASK_CC] ? PACK_IMG_ONE : PACK_IMG_M));
    Buf st = c.get(pair_bytes);
    int rc = run_layer(c, *pair1, stem_view(c, in8.p, H, W), st.p, 24, 0, 2);
    if (rc) return rc;
    c.put(in8);
    std::vector<std::string> na, nb;
    for (auto& n : trunk_rest) { na.push_back(n); nb.push_back("w" + n); }
    na.push_back("conv10_atrous"); nb.push_back("wconv10_atrous");
    rc = run_chain(c, 'G', na, pair_view(st.p, 0), false, Buf(), nullptr, nullptr, cat1.p, cat_ld, 0);
    if (rc) return rc;
    View v;
    Buf b;
    rc = run_chain(c, 'G', nb, pair_view(st.p, 1), false, Buf(), &v, &b);
    if (rc) return rc;
    c.put(st);
    Buf pooled = c.get((size_t)c.B * 96 * 4);
    c.tag("plane_reduce + broadcast_channels|global style pooling -> concat blocks", 0, 0, 0, 2.0 * c.B * h * w * 96 * (c.esz() > 2 ? 4 : 2));
    CK(do_pool_broadcast(c, v, h * w, opt[SE_OPT_POOL_AVG] ? RED_AVG : RED_MAX, (float*)pooled.p, cat1.p, cat_ld, tc));
    c.put(pooled);
    c.put(b);
  } else {
  {
      Buf in8 = c.get((size_t)c.B * H * stem_wp(W) * 8 * e);
      c.tag("pack8_kernel|mask-mul + concat + cast", 0, 0, 0, (double)c.B * H * W * 20 + (double)c.B * H * stem_wp(W) * 8 * c.esz());
      CK(do_pack8(c, x, guide, mask, in8.p, H, W, PACK_IMG_ONE_MINUS_M, 1.0f, 1));
      std::vector<std::string> names = with_prefix("", kTrunk9);
      names.push_back("conv10_atrous");
      int rc = run_chain(c, 'G', names, stem_view(c, in8.p, H, W), true, in8, nullptr, nullptr, cat1.p, cat_ld, 0);
      if (rc) return rc;
    }
    {
      Buf in8 = c.get((size_t)c.B * H * stem_wp(W) * 8 * e);
      c.tag("pack8_kernel|mask-mul + concat + cast", 0, 0, 0, (double)c.B * H * W * 20 + (double)c.B * H * stem_wp(W) * 8 * c.esz());
      CK(do_pack8(c, x2, guide, mask2, in8.p, H, W, opt[SE_OPT_NO_MASK_CC] ? PACK_IMG_ONE : PACK_IMG_M, opt[SE_OPT_JOINT_TRAIN_INP] ? 0.0f : 1.0f, 1));
      std::vector<std::string> names = with_prefix("w", kTrunk9);
      names.push_back("wconv10_atrous");
      View v;
      Buf b;
      int rc = run_chain(c, 'G', names, stem_view(c, in8.p, H, W), true, in8, &v, &b);
      if (rc) return rc;
      Buf pooled = c.get((size_t)c.B * 96 * 4);
      c.tag("plane_reduce + broadcast_channels|global style pooling -> concat blocks", 0, 0, 0, 2.0 * c.B * h * w * 96 * (c.esz() > 2 ? 4 : 2));
      CK(do_pool_broadcast(c, v, h * w, opt[SE_OPT_POOL_AVG] ? RED_AVG : RED_MAX, (float*)pooled.p, cat1.p, cat_ld, tc));
      c.put(pooled);
      c.put(b);
    }
  }
  Buf xnow = c.get((size_t)c.B * H * stem_wp(W) * 8 * e);
  {
    View v16;
    Buf b16;
    int rc = run_chain(c, 'G', with_prefix("conv", {"11", "12", "13_upsample_conv", "14", "15_upsample_conv", "16"}),
                       cat_view(cat1.p), true, cat1, &v16, &b16);
    if (rc) return rc;
    c.tag("memset|pad pixels of the packed stage-2 input", 0, 0, 0, (double)xnow.bytes);
    CK(fill_zero(xnow.p, xnow.bytes, c.stream));   // zero pad pixels of the packed stage-2 input
    rc = run_head(c, 'G', "conv17", v16, HEAD_COARSE, x, mask, nullptr, x_stage1, nullptr, xnow.p);
    if (rc) return rc;
    c.put(b16);
  }
  // ---- stage 2: hallucination branch + patch-match branch -> concat -> joint decoder
  Buf cat2 = c.get((size_t)c.B * h * w * 192 * e);
  Buf st2;
  if (pair2) {
    st2 = c.get(pair_bytes);
    int rc = run_layer(c, *pair2, stem_view(c, xnow.p, H, W), st2.p, 24, 0, 2);
    if (rc) return rc;
    c.put(xnow);
    std::vector<std::string> nx;
    for (auto& n : trunk_rest) nx.push_back("x" + n);
    nx.push_back("xconv10_atrous");
    rc = run_chain(c, 'G', nx, pair_view(st2.p, 0), false, Buf(), nullptr, nullptr, cat2.p, cat_ld, 0);
    if (rc) return rc;
  } else {
    std::vector<std::string> names = with_prefix("x", kTrunk9);
    names.push_back("xconv10_atrous");
    int rc = run_chain(c, 'G', names, stem_view(c, xnow.p, H, W), false, Buf(), nullptr, nullptr, cat2.p, cat_ld, 0);
    if (rc) return rc;
  }
  {
    View pm;
    Buf pmb;
    // pmconv6 writes the layout the attention reads: space-to-depth channel-blocked on the tensor-core path, NHWC otherwise
    const int pm_c8 = opt[SE_OPT_USE_CAM] ? (c.split() ? 1 : (tc ? 2 : 0)) : -1;
    int rc = pair2 ? run_chain(c, 'G', with_prefix("pm", {"conv2_downsample", "conv3", "conv4_downsample", "conv5", "conv6"}), pair_view(st2.p, 1), true, st2,
                               &pm, &pmb, nullptr, 0, 0, pm_c8)
                   : run_chain(c, 'G', with_prefix("pm", {"conv1", "conv2_downsample", "conv3", "conv4_downsample", "conv5", "conv6"}),
                               stem_view(c, xnow.p, H, W), true, xnow, &pm, &pmb, nullptr, 0, 0, pm_c8);
    if (rc) return rc;
    if (opt[SE_OPT_USE_CAM]) {
      Buf ms = c.get((size_t)c.B * h * w * 4);
      c.tag("avgpool4_kernel", 0, 0, 0, (double)c.B * H * W * 4);
      CK(avgpool4(mask, (float*)ms.p, c.B, H, W, c.stream));
      Buf camo = c.get((size_t)c.B * h * w * 96 * e);
      if (c.split()) {
        // split-half mode: fp32 NHWC in / out of the attention (split-half fp16 GEMMs over explicit patch matrices, se_gemm_split.cu)
        Buf f32 = c.get((size_t)c.B * h * w * 96 * 4), o32 = c.get((size_t)c.B * h * w * 96 * 4);
        CK(split_to_f32(pm.p, (float*)f32.p, c.B, 96, h * w, pm.ld / 2, 0, 1, c.stream));
        rc = run_cam_split(c, (const float*)f32.p, h, w, 96, (const float*)ms.p, (float*)o32.p);
        if (rc) return rc;
        CK(nhwc_f32_to_split((const float*)o32.p, camo.p, c.B, 96, h * w, 12, 0, c.stream));
        c.put(o32); c.put(f32);
      } else {
        rc = tc ? run_cam_tc(c, pm, (const float*)ms.p, camo.p, nullptr) : run_cam(c, pm, (const float*)ms.p, camo.p, 96, nullptr, 0);
        if (rc) return rc;
      }
      c.put(ms);
      c.put(pmb);
      pm = tc ? c8view(camo.p, h, w, 96, 12 * c.sp(), 0) : nhwc(camo.p, h, w, 96, 96);
      pmb = camo;
    }
    rc = run_chain(c, 'G', with_prefix("pm", {"conv9", "conv10"}), pm, true, pmb, nullptr, nullptr, cat2.p, cat_ld, 96);
    if (rc) return rc;
  }
  {
    View v16;
    Buf b16;
    int rc = run_chain(c, 'G', with_prefix("allconv", {"11", "12", "13_upsample_conv", "14", "15_upsample_conv", "16"}),
                       cat_view(cat2.p), true, cat2, &v16, &b16);
    if (rc) return rc;
    if (composed || composed_u8) {
      rc = run_head(c, 'G', "allconv17", v16, HEAD_FINE, blend_img, nullptr, mask_soft, composed, x_stage2, nullptr, composed_bs, msoft_bs, composed_u8);
    } else {
      rc = run_head(c, 'G', "allconv17", v16, HEAD_TANH, nullptr, nullptr, nullptr, x_stage2, nullptr, nullptr);
    }
    if (rc) return rc;
    c.put(b16);
  }
  return 0;
}

// run `fn` twice: dry (arena peak) then for real
static const bool g_graphs_on = getenv("SE_NO_GRAPHS") == nullptr;
static const bool g_graph_log = getenv("SE_GRAPH_LOG") != nullptr;   // one stderr line per capture / failed capture
constexpr size_t kMaxGraphs = 16;

template <typename F>
static int with_arena(se_model* m, int prec, int B, cudaStream_t stream, F fn, std::vector<uintptr_t> key = {}) {
  SE_REQUIRE(m && m->finalized, "model not finalized");
  SE_REQUIRE(prec >= 0 && prec <= 3, "precision");
  std::lock_guard<std::mutex> model_lock(m->mu);
  {
    int dev = -1;
    SE_CUDA_OK(cudaGetDevice(&dev));
    if (m->device < 0) m->device = dev;   // model-less operator holder: bound at first use
    SE_REQUIRE(dev == m->device, "model lives on device " + std::to_string(m->device) + " but the current device is " + std::to_string(dev));
    if (m->used && m->last_stream != stream) {
      // the previous forward may still be using the workspace on its own stream: order this one after it
      if (!m->order_ev) SE_CUDA_OK(cudaEventCreateWithFlags(&m->order_ev, cudaEventDisableTiming));
      SE_CUDA_OK(cudaEventRecord(m->order_ev, m->last_stream));
      SE_CUDA_OK(cudaStreamWaitEvent(stream, m->order_ev, 0));
    }
    m->last_stream = stream;
    m->used = true;
  }
  // ---- replay a captured forward
  const bool graphable = g_graphs_on && !g_timing && !key.empty() && getenv("SE_TC_DEBUG") == nullptr && getenv("SE_DEBUG_NAN") == nullptr;
  const bool legacy = (stream == nullptr || stream == cudaStreamLegacy);
  cudaStream_t gs = stream;   // stream the graph is captured on / launched into
  if (graphable && legacy) {
    if (!m->gstream) {
      SE_CUDA_OK(cudaStreamCreateWithFlags(&m->gstream, cudaStreamNonBlocking));
      SE_CUDA_OK(cudaEventCreateWithFlags(&m->bridge_in, cudaEventDisableTiming));
      SE_CUDA_OK(cudaEventCreateWithFlags(&m->bridge_out, cudaEventDisableTiming));
    }
    gs = m->gstream;
  }
  auto bridge_in = [&]() -> int {
    if (gs != stream) { SE_CUDA_OK(cudaEventRecord(m->bridge_in, stream)); SE_CUDA_OK(cudaStreamWaitEvent(gs, m->bridge_in, 0)); }
    return 0;
  };
  auto bridge_out = [&]() -> int {
    if (gs != stream) { SE_CUDA_OK(cudaEventRecord(m->bridge_out, gs)); SE_CUDA_OK(cudaStreamWaitEvent(stream, m->bridge_out, 0)); }
    return 0;
  };
  if (graphable) {
    for (int k = 0; k < 8; ++k) key.push_back((uintptr_t)m->opt[k]);
    key.push_back((uintptr_t)prec);
    key.push_back((uintptr_t)B);
    for (auto& g : m->graphs)
      if (g.exec && g.arena == m->arena && g.key == key) {
        int rb = bridge_in();
        if (rb) return rb;
        SE_CUDA_OK(cudaGraphLaunch(g.exec, gs));
        rb = bridge_out();
        if (rb) return rb;
        g.tick = ++m->tick;
        g_launches = g.launches;
        return 0;
      }
  }
  Ctx c;
  c.m = m; c.stream = stream; c.prec = prec; c.B = B;
  c.dry = true;
  c.arena.reset(nullptr);
  int rc = fn(c);
  if (rc) return rc;
  const size_t need = c.arena.peak + 4096;
  if (need > m->arena_bytes) {
    SE_CUDA_OK(cudaDeviceSynchronize());   // every stream that ever used the old slab
    for (auto& g : m->graphs) if (g.exec) cudaGraphExecDestroy(g.exec);   // captured on the old slab
    m->graphs.clear();
    if (m->arena) SE_CUDA_OK(cudaFree(m->arena));
    m->arena = nullptr;
    m->arena_bytes = 0;
    SE_CUDA_OK(cudaMalloc(&m->arena, need));
    m->arena_bytes = need;
  }
  c.dry = false;
  c.arena.reset((char*)m->arena);
  g_launches = 0;
  // ---- second sighting of this signature: capture the launches into a graph (first sighting runs eagerly: it also performs the
  // one-time initialisations - function attributes, driver entry points - that must not happen inside a capture)
  if (graphable && m->seen[key]++ >= 1) {
    cudaGraph_t graph = nullptr;
    int rb = bridge_in();
    if (rb) return rb;
    if (cudaStreamBeginCapture(gs, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
      c.stream = gs;
      rc = fn(c);
      c.stream = stream;
      const cudaError_t ce = cudaStreamEndCapture(gs, &graph);
      cudaGraphExec_t exec = nullptr;
      if (rc == 0 && ce == cudaSuccess && graph && cudaGraphInstantiate(&exec, graph, 0) == cudaSuccess) {
        cudaGraphDestroy(graph);
        if (m->graphs.size() >= kMaxGraphs) {   // evict the least recently used
          size_t lru = 0;
          for (size_t i = 1; i < m->graphs.size(); ++i) if (m->graphs[i].tick < m->graphs[lru].tick) lru = i;
          cudaGraphExecDestroy(m->graphs[lru].exec);
          m->graphs.erase(m->graphs.begin() + lru);
        }
        se_model::GraphEntry e;
        e.key = key; e.exec = exec; e.arena = m->arena; e.launches = g_launches; e.tick = ++m->tick;
        m->graphs.push_back(e);
        if (g_graph_log) fprintf(stderr, "[graph] captured B=%d prec=%d launches=%d (%zu cached)\n", B, prec, e.launches, m->graphs.size());
        SE_CUDA_OK(cudaGraphLaunch(exec, gs));
        return bridge_out();
      }
      if (g_graph_log) fprintf(stderr, "[graph] capture failed: rc=%d end=%s exec=%p\n", rc, cudaGetErrorString(ce), (void*)exec);
      if (graph) cudaGraphDestroy(graph);
      (void)cudaGetLastError();
      m->seen[key] = -1000000;   // not capturable: stay eager for this signature
      if (rc) return rc;
      c.arena.reset((char*)m->arena);
      g_launches = 0;
    } else {
      if (g_graph_log) fprintf(stderr, "[graph] cudaStreamBeginCapture failed: %s\n", cudaGetErrorString(cudaPeekAtLastError()));
      (void)cudaGetLastError();  // a failed cudaStreamBeginCapture leaves a sticky error behind
      m->seen[key] = -1000000;
    }
    rb = bridge_out();           // (orders nothing new, but keeps the two streams' event pairs balanced)
    if (rb) return rb;
  }
  if (g_graph_log && graphable) fprintf(stderr, "[graph] eager run B=%d prec=%d (sighting %d of this signature, %zu signatures seen)\n", B, prec, m->seen[key], m->seen.size());
  return fn(c);
}

// Two 5x5 stems that read the SAME packed 8-channel input become ONE launch with N = 96 (a stem tile is bound by its per-tile
// protocol and the small-N MMA rate, not by math: one N = 96 launch costs about what one N = 48 launch does).
//   "G.conv1+wconv1": packed input [x(1-m) (3), sketch, m, x2*m2 (3)]: conv1 reads channels 0..4, wconv1 its own image copy in
//                     5..7, the sketch channel (weight zeroed under --joint_train_inp, where the reference feeds zeros) and m
//   "G.xconv1+pmconv1": both read the 3 channels of the blended coarse result
// Fused output channel order [fA(24) fB(24) | gA(24) gB(24)] so that it is an ordinary gated layer with 96 outputs; the epilogue
// sends output blocks 0-2 to layer A's space-to-depth tensor and blocks 3-5 to layer B's (EpiParams::blk_split).
static int make_stem_pair(se_model* m, const char* key, const char* a, const char* b, const int* chan_a, const int* chan_b, float scale_b3) {
  Layer* A = find_layer(m, 'G', a);
  Layer* B = find_layer(m, 'G', b);
  if (!A || !B || !A->set || !B->set) return 0;
  Layer F;
  F.name = key;
  F.spec = Spec{nullptr, 8, 96, 5, 1, 1, false, 0};
  F.set = true;
  F.fused_pair = true;
  F.pair_cin_sum = A->spec.cin + B->spec.cin;
  F.w_host.assign((size_t)96 * 8 * 25, 0.0f);
  F.b_host.assign(96, 0.0f);
  for (int n = 0; n < 96; ++n) {
    const bool gate = n >= 48;
    const int r = n % 48;
    const Layer* S = r < 24 ? A : B;
    const int* chan = r < 24 ? chan_a : chan_b;
    const int co = (r % 24) + (gate ? 24 : 0);           // channel of the source layer: features 0..23, gates 24..47
    F.b_host[n] = S->b_host[co];
    for (int ci = 0; ci < S->spec.cin; ++ci) {
      const float sc = (S == B && ci == 3) ? scale_b3 : 1.0f;
      for (int t = 0; t < 25; ++t) F.w_host[((size_t)n * 8 + chan[ci]) * 25 + t] = S->w_host[((size_t)co * S->spec.cin + ci) * 25 + t] * sc;
    }
  }
  int rc = pack_layer(m, F);
  if (rc) return rc;
  F.w_host.clear();
  m->layers[std::string("G.") + key] = F;
  return 0;
}

static int check_hw(int H, int W) {
  SE_REQUIRE(H % 8 == 0 && W % 8 == 0 && H >= 16 && W >= 16, "H and W must be multiples of 8 and >= 16 (two stride-2 convs, 4x4 mask pool, stride-2 patch grid)");
  return 0;
}

}  // namespace se

// ============================================================================================ C ABI
extern "C" {

const char* se_last_error(void) { return se::last_error(); }
int se_abi_version(void) { return 1; }

int se_model_create(se_model** out) {
  SE_REQUIRE(out != nullptr, "out");
  se_model* m = new se_model();
  for (char net : {'M', 'G'}) {
    ArchTable t = make_arch(net);
    for (size_t i = 0; i < t.specs.size(); ++i) {
      Layer L;
      L.spec = t.specs[i];
      L.name = t.names[i];
      m->layers[std::string(1, net) + "." + t.names[i]] = L;
    }
  }
  *out = m;
  return 0;
}

void se_model_destroy(se_model* m) {
  if (!m) return;
  for (void* p : m->owned) cudaFree(p);
  if (m->arena) cudaFree(m->arena);
  if (m->order_ev) cudaEventDestroy(m->order_ev);
  for (auto& g : m->graphs) if (g.exec) cudaGraphExecDestroy(g.exec);
  if (m->gstream) cudaStreamDestroy(m->gstream);
  if (m->bridge_in) cudaEventDestroy(m->bridge_in);
  if (m->bridge_out) cudaEventDestroy(m->bridge_out);
  delete m;
}

int se_model_set_layer(se_model* m, char net, const char* layer, const float* weight, const float* bias, int cout, int cin, int ksize) {
  SE_REQUIRE(m && layer && weight && bias, "null argument");
  SE_REQUIRE(!m->finalized, "model already finalized");
  Layer* L = find_layer(m, net, layer);
  SE_REQUIRE(L != nullptr, std::string("no such layer: net") + net + "." + layer);
  SE_REQUIRE(L->spec.cout == cout && L->spec.cin == cin && L->spec.k == ksize,
             std::string("shape mismatch for ") + layer + ": expected [" + std::to_string(L->spec.cout) + "," + std::to_string(L->spec.cin) + "," +
                 std::to_string(L->spec.k) + "," + std::to_string(L->spec.k) + "]");
  L->w_host.assign(weight, weight + (size_t)cout * cin * ksize * ksize);
  L->b_host.assign(bias, bias + cout);
  L->set = true;
  return 0;
}

int se_model_set_option(se_model* m, int option, int value) {
  SE_REQUIRE(m && option >= 0 && option < 8, "option");
  SE_REQUIRE(!m->finalized, "options are fixed at se_model_finalize (they shape the packed weights)");
  m->opt[option] = value;
  return 0;
}

int se_model_finalize(se_model* m) {
  SE_REQUIRE(m, "model");
  SE_REQUIRE(!m->finalized, "model already finalized");
  int ndev = 0;
  SE_CUDA_OK(cudaGetDeviceCount(&ndev));
  SE_REQUIRE(ndev > 0, "no CUDA device: sketchedit_b200 has no CPU fallback");
  SE_CUDA_OK(cudaGetDevice(&m->device));   // packed weights and the workspace live on the device current now
  // a net may be left out entirely (stand-alone netM / netG modules); a partially set net is an error
  for (char net : {'M', 'G'}) {
    int nset = 0, ntot = 0;
    std::string first_missing;
    for (auto& kv : m->layers)
      if (kv.first[0] == net) {
        ++ntot;
        if (kv.second.set) ++nset;
        else if (first_missing.empty()) first_missing = kv.first;
      }
    SE_REQUIRE(nset == 0 || nset == ntot, "layer not set: net" + first_missing);
  }
  {
    static const bool no_pairs = getenv("SE_NO_STEM_PAIRS") != nullptr;   // A/B switch for experiments
    const int id5[5] = {0, 1, 2, 3, 4}, w5[5] = {5, 6, 7, 3, 4}, id3[3] = {0, 1, 2};
    if (!no_pairs) {
      int rc = make_stem_pair(m, "conv1+wconv1", "conv1", "wconv1", id5, w5, m->opt[SE_OPT_JOINT_TRAIN_INP] ? 0.0f : 1.0f);
      if (rc) return rc;
      rc = make_stem_pair(m, "xconv1+pmconv1", "xconv1", "pmconv1", id3, id3, 1.0f);
      if (rc) return rc;
    }
  }
  for (auto& kv : m->layers) {
    if (!kv.second.set || kv.second.fused_pair) continue;
    int rc = pack_layer(m, kv.second);
    if (rc) return rc;
    kv.second.w_host.clear();
    kv.second.w_host.shrink_to_fit();
  }
  m->finalized = true;
  return 0;
}

static int forward_inference(se_model* m, const float* image, const float* sketch, int B, int H, int W, int precision, float* composed,
                             float* mask, long long composed_bs, long long mask_bs, float* coarse, float* fine, float* mask_image,
                             const float* mask_bin_in, float* mask_bin_out, cudaStream_t st) {
  SE_REQUIRE(image && sketch && composed && mask, "null tensor");
  int rc = check_hw(H, W);
  if (rc) return rc;
  std::vector<uintptr_t> key = {1, (uintptr_t)H, (uintptr_t)W, (uintptr_t)image, (uintptr_t)sketch, (uintptr_t)composed, (uintptr_t)mask, (uintptr_t)composed_bs,
                                (uintptr_t)mask_bs, (uintptr_t)coarse, (uintptr_t)fine, (uintptr_t)mask_image, (uintptr_t)mask_bin_in, (uintptr_t)mask_bin_out};
  return with_arena(m, precision, B, st, [&](Ctx& c) -> int {
    Buf mb = c.get((size_t)B * H * W * 4);
    int r = run_netM(c, image, sketch, H, W, mask, mask_image, (float*)mb.p, mask_bs);
    if (r) return r;
    const float* mbin = (const float*)mb.p;
    if (mask_bin_in) mbin = mask_bin_in;
    if (mask_bin_out && !c.dry) {
      SE_CUDA_OK(cudaMemcpyAsync(mask_bin_out, mbin, (size_t)B * H * W * 4, cudaMemcpyDeviceToDevice, c.stream));
    }
    // generate_fake: netG(inputs, inputs, mask_bin, mask_bin, line)   (editline2_model.py:368)
    r = run_netG(c, image, image, mbin, mbin, sketch, H, W, coarse, fine, composed, mask, image, composed_bs, mask_bs);
    if (r) return r;
    c.put(mb);
    return 0;
  }, key);
}

int se_forward_inference(se_model* m, const float* image, const float* sketch, int B, int H, int W, int precision, float* composed,
                         float* mask, float* coarse, float* fine, float* mask_image, const float* mask_bin_in, float* mask_bin_out,
                         void* stream) {
  return forward_inference(m, image, sketch, B, H, W, precision, composed, mask, 0, 0, coarse, fine, mask_image, mask_bin_in, mask_bin_out,
                           (cudaStream_t)stream);
}

int se_forward_inference_packed(se_model* m, const float* image, const float* sketch, int B, int H, int W, int precision, float* packed,
                                void* stream) {
  SE_REQUIRE(packed != nullptr, "null tensor");
  const long long bs = 4LL * H * W;   // [B,4,H,W]: composed in channels 0-2, the soft mask in channel 3
  return forward_inference(m, image, sketch, B, H, W, precision, packed, packed + 3LL * H * W, bs, bs, nullptr, nullptr, nullptr, nullptr, nullptr,
                           (cudaStream_t)stream);
}

int se_forward_inference_u8(se_model* m, const unsigned char* image_u8, const unsigned char* sketch_u8, int B, int H, int W, int precision,
                            unsigned char* bgr_u8, unsigned char* mask_u8, void* stream) {
  SE_REQUIRE(image_u8 && sketch_u8 && bgr_u8 && mask_u8, "null tensor");
  int rc = check_hw(H, W);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  std::vector<uintptr_t> key = {4, (uintptr_t)H, (uintptr_t)W, (uintptr_t)image_u8, (uintptr_t)sketch_u8, (uintptr_t)bgr_u8, (uintptr_t)mask_u8};
  return with_arena(m, precision, B, st, [&](Ctx& c) -> int {
    // input codec (reference data/testimage_dataset.py:89-103) -> the usual forward -> output codec fused into the two heads
    // (test.py:25-35): the float image / masks live only in the workspace
    Buf img = c.get((size_t)B * 3 * H * W * 4), sk = c.get((size_t)B * H * W * 4), soft = c.get((size_t)B * H * W * 4), mb = c.get((size_t)B * H * W * 4);
    c.tag("u8_to_inputs_kernel|input codec", 0, 0, 0, (double)B * H * W * (4 + 16));
    CK(u8_to_inputs(image_u8, sketch_u8, (float*)img.p, (float*)sk.p, B, H, W, c.stream));
    int r = run_netM(c, (const float*)img.p, (const float*)sk.p, H, W, (float*)soft.p, nullptr, (float*)mb.p, 0, mask_u8);
    if (r) return r;
    r = run_netG(c, (const float*)img.p, (const float*)img.p, (const float*)mb.p, (const float*)mb.p, (const float*)sk.p, H, W, nullptr, nullptr, nullptr,
                 (const float*)soft.p, (const float*)img.p, 0, 0, bgr_u8);
    if (r) return r;
    c.put(mb); c.put(soft); c.put(sk); c.put(img);
    return 0;
  }, key);
}

// generate_fake's external-mask branch at inference (editline2_model.py:343-345,362-368): netG(x, x, R, R, s*R), composed with R
// (:114); netM does not run. The final head's blend with R in place of the soft mask leaves x bit for bit where R = 0.
int se_forward_inpaint(se_model* m, const float* image, const float* sketch, const float* region, int B, int H, int W, int precision,
                       float* composed, float* coarse, float* fine, void* stream) {
  SE_REQUIRE(image && sketch && region && composed, "null tensor");
  int rc = check_hw(H, W);
  if (rc) return rc;
  std::vector<uintptr_t> key = {5, (uintptr_t)H, (uintptr_t)W, (uintptr_t)image, (uintptr_t)sketch, (uintptr_t)region, (uintptr_t)composed,
                                (uintptr_t)coarse, (uintptr_t)fine};
  return with_arena(m, precision, B, (cudaStream_t)stream, [&](Ctx& c) -> int {
    Buf sr = c.get((size_t)B * H * W * 4);
    c.tag("region_inputs_kernel|sketch * region", 0, 0, 0, (double)B * H * W * 12);
    CK(region_sketch(sketch, region, (float*)sr.p, B, H, W, c.stream));
    int r = run_netG(c, image, image, region, region, (const float*)sr.p, H, W, coarse, fine, composed, region, image);
    if (r) return r;
    c.put(sr);
    return 0;
  }, key);
}

int se_forward_inpaint_u8(se_model* m, const unsigned char* image_u8, const unsigned char* sketch_u8, const unsigned char* region_u8, int B, int H,
                          int W, int precision, unsigned char* bgr_u8, void* stream) {
  SE_REQUIRE(image_u8 && sketch_u8 && region_u8 && bgr_u8, "null tensor");
  int rc = check_hw(H, W);
  if (rc) return rc;
  std::vector<uintptr_t> key = {6, (uintptr_t)H, (uintptr_t)W, (uintptr_t)image_u8, (uintptr_t)sketch_u8, (uintptr_t)region_u8, (uintptr_t)bgr_u8};
  return with_arena(m, precision, B, (cudaStream_t)stream, [&](Ctx& c) -> int {
    // input codec (the sketch's, data/testimage_dataset.py:89-103, also for the region) -> netG -> output codec fused into the last head
    Buf img = c.get((size_t)B * 3 * H * W * 4), rg = c.get((size_t)B * H * W * 4), sr = c.get((size_t)B * H * W * 4);
    c.tag("region_inputs_kernel|input codec + sketch * region", 0, 0, 0, (double)B * H * W * (5 + 20));
    CK(region_inputs_u8(image_u8, sketch_u8, region_u8, (float*)img.p, (float*)rg.p, (float*)sr.p, B, H, W, c.stream));
    const float* x = (const float*)img.p;
    const float* R = (const float*)rg.p;
    int r = run_netG(c, x, x, R, R, (const float*)sr.p, H, W, nullptr, nullptr, nullptr, R, x, 0, 0, bgr_u8);
    if (r) return r;
    c.put(sr); c.put(rg); c.put(img);
    return 0;
  }, key);
}

int se_netM_forward(se_model* m, const float* x, const float* guide, int B, int H, int W, int precision, float* mask1, float* x_stage1,
                    void* stream) {
  SE_REQUIRE(x && guide && mask1, "null tensor");
  int rc = check_hw(H, W);
  if (rc) return rc;
  return with_arena(m, precision, B, (cudaStream_t)stream, [&](Ctx& c) -> int { return run_netM(c, x, guide, H, W, mask1, x_stage1, nullptr); },
                    {2, (uintptr_t)H, (uintptr_t)W, (uintptr_t)x, (uintptr_t)guide, (uintptr_t)mask1, (uintptr_t)x_stage1});
}

int se_netG_forward(se_model* m, const float* x, const float* x2, const float* mask, const float* mask2, const float* guide, int B, int H,
                    int W, int precision, float* x_stage1, float* x_stage2, void* stream) {
  SE_REQUIRE(x && x2 && mask && mask2 && x_stage2, "null tensor");   // guide may be NULL: guide=None of the reference
  int rc = check_hw(H, W);
  if (rc) return rc;
  return with_arena(m, precision, B, (cudaStream_t)stream,
                    [&](Ctx& c) -> int { return run_netG(c, x, x2, mask, mask2, guide, H, W, x_stage1, x_stage2, nullptr, nullptr, nullptr); },
                    {3, (uintptr_t)H, (uintptr_t)W, (uintptr_t)x, (uintptr_t)x2, (uintptr_t)mask, (uintptr_t)mask2, (uintptr_t)guide, (uintptr_t)x_stage1, (uintptr_t)x_stage2});
}

int se_gated_conv_forward(se_model* m, char net, const char* layer, const float* x, int B, int H, int W, int precision, float* y,
                          void* stream) {
  SE_REQUIRE(m && layer && x && y, "null argument");
  Layer* L = find_ready(m, net, layer);
  SE_REQUIRE(L != nullptr, std::string("no such (loaded) layer: ") + layer);
  cudaStream_t st = (cudaStream_t)stream;
  // heads are raw fp32 CUDA-core convolutions in every mode; the fp32-on-tensor-cores mode runs them like the fp32 path
  if (precision == SE_PREC_FP32_TC && L->is_head) precision = SE_PREC_FP32_EXACT;
  return with_arena(m, precision, B, st, [&](Ctx& c) -> int {
    const Spec& s = L->spec;
    const int dt = c.act_dt();
    const int Ci = L->is_head ? 12 : L->Ci;
    const int in_c8 = wants_c8(c, *L);
    Buf in = c.get(L->is_stem ? (size_t)B * H * stem_wp(W) * 8 * c.esz() : act_bytes(c, H, W, Ci, in_c8));
    if (c.split()) {
      // split-half storage: hi / lo fp16 halves of the fp32 input in the layout the layer reads
      if (L->is_stem || s.cin % 8) CK(fill_zero(in.p, in.bytes, c.stream));
      CK(nchw_to_split(x, in.p, B, s.cin, H, W, L->is_stem ? 3 : in_c8, stem_wp(W), STEM_PADL, c.stream));
    } else if (L->is_stem) {
      CK(fill_zero(in.p, in.bytes, c.stream));
      CK(nchw_to_stem8(x, in.p, dt, B, s.cin, H, W, stem_wp(W), STEM_PADL, c.stream));
    } else if (in_c8 == 2) {
      CK(nchw_to_c8_s2d(x, in.p, B, s.cin, H, W, c.stream));
    } else if (in_c8) {
      if (s.cin % 8) CK(fill_zero(in.p, in.bytes, c.stream));
      CK(nchw_to_c8(x, in.p, B, s.cin, H * W, c.stream));
    } else {
      CK(nchw_to_nhwc(x, in.p, dt, B, s.cin, H * W, Ci, 0, c.stream));
    }
    int Ho, Wo;
    out_dims(s, H, W, &Ho, &Wo);
    if (L->is_head) {
      // raw conv (activation=None / cout==3, utils.py:27): run through the direct kernel, fp32 out
      Buf o = c.get((size_t)B * Ho * Wo * s.cout * 4);
      ConvParams cp;
      memset(&cp, 0, sizeof(cp));
      ClassW& cw = L->cls[0];
      cp.x = in.p; cp.in_dt = dt; cp.N = B; cp.Hi = H; cp.Wi = W; cp.Ci = Ci; cp.ldx = Ci;
      cp.Ho = Ho; cp.Wo = Wo; cp.stride = 1; cp.ntaps = cw.ntaps;
      memcpy(cp.dy, cw.dy, sizeof(cp.dy));
      memcpy(cp.dx, cw.dx, sizeof(cp.dx));
      cp.w = cw.w_direct; cp.bias = L->bias; cp.Cout = s.cout;
      cp.y = o.p; cp.out_dt = DT_F32; cp.Hout = Ho; cp.Wout = Wo; cp.ldo = s.cout; cp.choff = 0;
      cp.osy = cp.osx = 1; cp.epi = EPI_LINEAR; cp.scale = 1.0f;
      CK(direct_launch(cp, cw.CoutP, precision == SE_PREC_FP32_EXACT, c.stream));
      CK(nhwc_to_nchw(o.p, DT_F32, y, B, s.cout, Ho * Wo, s.cout, 0, c.stream));
      c.put(o);
    } else {
      const int cg = s.cout / 2;
      View vin = L->is_stem ? stem_view(c, in.p, H, W) : (in_c8 ? c8view(in.p, H, W, Ci, (Ci + 7) / 8 * c.sp(), 0) : nhwc(in.p, H, W, Ci, Ci));
      if (in_c8 == 2) { vin.c8 = 2; vin.ld = 4 * (Ci / 8) * c.sp(); }
      if (c.split()) {
        const int cbo = (cg + 7) / 8;
        Buf o = c.get(act_bytes(c, Ho, Wo, cg, 1));
        if (cg % 8) CK(fill_zero(o.p, o.bytes, c.stream));
        int r = run_layer(c, *L, vin, o.p, 2 * cbo, 0, 1);
        if (r) return r;
        CK(split_to_f32(o.p, y, B, cg, Ho * Wo, cbo, 0, 0, c.stream));
        c.put(o);
      } else {
        Buf o = c.get((size_t)B * Ho * Wo * cg * c.esz());
        int r = run_layer(c, *L, vin, o.p, cg, 0, 0);
        if (r) return r;
        CK(nhwc_to_nchw(o.p, dt, y, B, cg, Ho * Wo, cg, 0, c.stream));
        c.put(o);
      }
    }
    c.put(in);
    return 0;
  });
}

int se_contextual_attention_forward(const float* feat, const float* mask_s, int B, int C, int h, int w, int precision, float* out,
                                    float* attn, void* stream) {
  SE_REQUIRE(feat && mask_s && out, "null tensor");
  static se_model* holder = nullptr;   // arena owner for the model-less operator call
  static std::mutex mu;
  std::lock_guard<std::mutex> lk(mu);
  if (!holder) { holder = new se_model(); holder->finalized = true; }
  // fp32-on-tensor-cores mode: split-half GEMM attention (needs 16 * C to be a multiple of 256 and no attention-map output);
  // everything else of the fp32 modes runs on the fp32 CUDA-core kernels
  const bool split_cam = precision == SE_PREC_FP32_TC && C % 16 == 0 && attn == nullptr && h % 2 == 0 && w % 2 == 0;
  if (precision == SE_PREC_FP32_TC) precision = SE_PREC_FP32_EXACT;
  cudaStream_t st = (cudaStream_t)stream;
  return with_arena(holder, precision, B, st, [&](Ctx& c) -> int {
    const int dt = c.act_dt();
    if (split_cam) {
      Buf in = c.get((size_t)B * h * w * C * 4), o = c.get((size_t)B * h * w * C * 4);
      CK(nchw_to_nhwc(feat, in.p, DT_F32, B, C, h * w, C, 0, c.stream));
      int r = run_cam_split(c, (const float*)in.p, h, w, C, mask_s, (float*)o.p);
      if (r) return r;
      CK(nhwc_to_nchw(o.p, DT_F32, out, B, C, h * w, C, 0, c.stream));
      c.put(o);
      c.put(in);
      return 0;
    }
    Buf in = c.get((size_t)B * h * w * C * c.esz());
    Buf o = c.get((size_t)B * h * w * C * c.esz());
    if (precision == SE_PREC_BF16_TC && C == 96 && h % 2 == 0 && w % 2 == 0) {
      // the layouts netG uses on the tensor-core path: space-to-depth channel-blocked in, channel-blocked out
      CK(nchw_to_c8_s2d(feat, in.p, B, C, h, w, c.stream));
      View fv = c8view(in.p, h, w, C, 4 * (C / 8), 0);
      fv.c8 = 2;
      int r = run_cam_tc(c, fv, mask_s, o.p, attn);
      if (r) return r;
      CK(c8_to_nchw(o.p, out, B, C, h * w, c.stream));
      c.put(o);
      c.put(in);
      return 0;
    }
    CK(nchw_to_nhwc(feat, in.p, dt, B, C, h * w, C, 0, c.stream));
    int r = run_cam(c, nhwc(in.p, h, w, C, C), mask_s, o.p, C, attn);
    if (r) return r;
    CK(nhwc_to_nchw(o.p, dt, out, B, C, h * w, C, 0, c.stream));
    c.put(o);
    c.put(in);
    return 0;
  });
}

int se_outputs_to_uint8(const float* composed, const float* mask, int B, int H, int W, unsigned char* bgr_hwc, unsigned char* mask_u8,
                        void* stream) {
  SE_REQUIRE(composed && bgr_hwc && (mask || !mask_u8), "null tensor");
  return to_uint8(composed, mask, bgr_hwc, mask_u8, B, H, W, (cudaStream_t)stream);
}

int se_resize_u8(const unsigned char* src, const long long* src_off, const int* src_hw, int B, int C, unsigned char* dst,
                 const long long* dst_off, const int* dst_hw, int flags, void* stream) {
  SE_REQUIRE(src && src_off && src_hw && dst && dst_off && dst_hw, "null argument");
  SE_REQUIRE(B >= 1 && B <= 65535, "B must be in [1, 65535] (one grid row per image)");
  SE_REQUIRE(C == 1 || C == 3, "C must be 1 or 3");
  SE_REQUIRE((flags & ~SE_RESIZE_REVERSE_CHANNELS) == 0, "unknown flag");
  for (int i = 0; i < B; ++i) {
    const long long hi = src_hw[2 * i], wi = src_hw[2 * i + 1], ho = dst_hw[2 * i], wo = dst_hw[2 * i + 1];
    SE_REQUIRE(hi >= 1 && wi >= 1 && ho >= 1 && wo >= 1, "image " + std::to_string(i) + ": sizes must be positive");
    SE_REQUIRE(std::max(hi, ho) * std::max(wi, wo) * C < (1LL << 31), "image " + std::to_string(i) + ": too large");
    SE_REQUIRE(src_off[i] >= 0 && dst_off[i] >= 0, "image " + std::to_string(i) + ": negative offset");
  }
  // arena owner of the model-less operator, one per device (like se_contextual_attention_forward's)
  static std::mutex holders_mu;
  static std::map<int, se_model*> holders;
  int dev = -1;
  SE_CUDA_OK(cudaGetDevice(&dev));
  se_model* holder;
  {
    std::lock_guard<std::mutex> lk(holders_mu);
    se_model*& h = holders[dev];
    if (!h) { h = new se_model(); h->finalized = true; }
    holder = h;
  }
  const int rev = (flags & SE_RESIZE_REVERSE_CHANNELS) ? 1 : 0;
  return with_arena(holder, SE_PREC_BF16_TC, B, (cudaStream_t)stream, [&](Ctx& c) -> int {
    // scratch: the jobs of both passes, then the uint8 intermediate of every image whose width AND height change
    std::vector<size_t> tmp_off(B, 0);
    size_t tmp_bytes = 0;
    for (int i = 0; i < B; ++i)
      if (src_hw[2 * i] != dst_hw[2 * i] && src_hw[2 * i + 1] != dst_hw[2 * i + 1]) {
        tmp_off[i] = tmp_bytes;
        tmp_bytes += ((size_t)src_hw[2 * i] * dst_hw[2 * i + 1] * C + 255) / 256 * 256;
      }
    Buf jb = c.get((size_t)2 * B * sizeof(ResizeJob));
    Buf tmp = c.get(tmp_bytes);
    if (!c.dry) {
      std::vector<ResizeJob> hj, vj;
      long long hmax = 0, vmax = 0;
      for (int i = 0; i < B; ++i) {
        const int hi = src_hw[2 * i], wi = src_hw[2 * i + 1], ho = dst_hw[2 * i], wo = dst_hw[2 * i + 1];
        const unsigned char* in = src + src_off[i];
        unsigned char* out = dst + dst_off[i];
        if (wi != wo || hi == ho) {   // horizontal pass, or the copy of an unchanged size
          ResizeJob j{in, hi != ho ? (unsigned char*)tmp.p + tmp_off[i] : out, nullptr, nullptr, 0, wi, hi, wo, hi != ho ? 0 : rev};
          if (wi != wo) {
            ResizeTable t;
            int r = resize_table(wi, wo, c.stream, &t);
            if (r) return r;
            j.bounds = t.bounds; j.weights = t.weights; j.ksize = t.ksize;
          }
          hj.push_back(j);
          hmax = std::max(hmax, (long long)hi * wo);
          if (hi != ho) in = j.out;
        }
        if (hi != ho) {
          ResizeTable t;
          int r = resize_table(hi, ho, c.stream, &t);
          if (r) return r;
          vj.push_back(ResizeJob{in, out, t.bounds, t.weights, t.ksize, wo, ho, wo, rev});
          vmax = std::max(vmax, (long long)ho * wo);
        }
      }
      const size_t nh = hj.size();
      hj.insert(hj.end(), vj.begin(), vj.end());
      SE_CUDA_OK(cudaMemcpyAsync(jb.p, hj.data(), hj.size() * sizeof(ResizeJob), cudaMemcpyHostToDevice, c.stream));
      const ResizeJob* jobs = (const ResizeJob*)jb.p;
      if (nh) CK(resize_pass(jobs, (int)nh, hmax, C, 0, c.stream));
      if (!vj.empty()) CK(resize_pass(jobs + nh, (int)vj.size(), vmax, C, 1, c.stream));
    }
    c.put(tmp);
    c.put(jb);
    return 0;
  });
}

int se_resize_coeffs(int in, int out, int* bounds, int* weights, int cap) {
  if (in < 1 || out < 1) {
    se::set_error("se_resize_coeffs: sizes must be positive");
    return -1;
  }
  std::vector<int> b, w;
  const int ksize = resize_coeffs(in, out, b, w);
  if (bounds && weights && (long long)cap >= (long long)w.size()) {
    memcpy(bounds, b.data(), b.size() * sizeof(int));
    memcpy(weights, w.data(), w.size() * sizeof(int));
  }
  return ksize;
}

int se_last_launch_count(void) { return se::g_launches; }
long long se_workspace_bytes(se_model* m) { return m ? (long long)m->arena_bytes : 0; }

int se_timing_enable(int on) {
  std::lock_guard<std::mutex> lk(g_time_mu);
  g_timing = on != 0;
  g_tl_used = 0;
  g_classes.clear();
  g_class_idx.clear();
  return 0;
}

// JSON text: {"classes":[{"name","tensor","launches","ms","flops_alg","flops_exec","bytes_alg"},...]} of everything
// launched since se_timing_enable(1). Synchronises on the recorded events. Returns the length needed (>= cap: truncated).
int se_timing_report(char* buf, int cap) {
  std::lock_guard<std::mutex> lk(g_time_mu);
  for (auto& a : g_classes) a.ms = 0.0;
  for (size_t i = 0; i < g_tl_used; ++i) {
    float t = 0.0f;
    if (cudaEventSynchronize(g_tl[i].b) != cudaSuccess || cudaEventElapsedTime(&t, g_tl[i].a, g_tl[i].b) != cudaSuccess) {
      set_error("se_timing_report: event query failed");
      return -1;
    }
    g_classes[g_tl[i].cls].ms += t;
  }
  std::string out = "{\"classes\":[";
  for (size_t i = 0; i < g_classes.size(); ++i) {
    const ClassAgg& a = g_classes[i];
    char num[256];
    snprintf(num, sizeof(num), "\",\"tensor\":%d,\"launches\":%d,\"ms\":%.6f,\"flops_alg\":%.6e,\"flops_exec\":%.6e,\"bytes_alg\":%.6e}", a.tensor, a.launches,
             a.ms, a.flops_alg, a.flops_exec, a.bytes_alg);
    out += std::string(i ? "," : "") + "{\"name\":\"" + a.name + num;
  }
  out += "]}";
  if (buf && cap > 0) {
    const size_t n = out.size() < (size_t)cap - 1 ? out.size() : (size_t)cap - 1;
    memcpy(buf, out.data(), n);
    buf[n] = 0;
  }
  return (int)out.size() + 1;
}

}  // extern "C"
