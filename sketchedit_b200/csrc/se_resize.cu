// Pillow's Image.resize with its default filter (BICUBIC) on uint8 HWC images, bit for bit: the serving path's resize to a
// multiple of 8 and back (reference demo.py:45,49,68). Pillow: src/libImaging/Resample.c (precompute_coeffs,
// normalize_coeffs_8bpc, ImagingResampleHorizontal_8bpc / Vertical_8bpc); oracle/pil_resample.py restates it in numpy.
//
// The coefficient tables are built on the host in double precision. This file is compiled with -ffp-contract=off
// (sketchedit_b200/build.py): a fused multiply-add changes the last bit of a weight, and that can move its fixed-point value.
#include <array>
#include <cmath>
#include <map>
#include <mutex>

#include "se_resize.h"

namespace se {

constexpr int kResizeBits = 22;   // Pillow's PRECISION_BITS for 8-bit images (32 - 8 - 2)

static double bicubic(double x) {
  const double a = -0.5;
  if (x < 0.0) x = -x;
  if (x < 1.0) return ((a + 2.0) * x - (a + 3.0)) * x * x + 1;
  if (x < 2.0) return (((x - 5) * x + 8) * x - 4) * a;
  return 0.0;
}

int resize_coeffs(int in, int out, std::vector<int>& bounds, std::vector<int>& weights) {
  const double scale = (double)in / out;
  const double fs = scale < 1.0 ? 1.0 : scale;
  const double support = 2.0 * fs;
  const int ksize = (int)std::ceil(support) * 2 + 1;
  bounds.assign((size_t)out * 2, 0);
  weights.assign((size_t)out * ksize, 0);
  std::vector<double> k(ksize);
  for (int xx = 0; xx < out; ++xx) {
    const double center = (xx + 0.5) * scale;
    const double ss = 1.0 / fs;
    int xmin = (int)(center - support + 0.5);
    if (xmin < 0) xmin = 0;
    int xmax = (int)(center + support + 0.5);
    if (xmax > in) xmax = in;
    xmax -= xmin;
    double ww = 0.0;
    for (int x = 0; x < xmax; ++x) {
      k[x] = bicubic((x + xmin - center + 0.5) * ss);
      ww += k[x];
    }
    for (int x = 0; x < xmax; ++x) {
      double w = k[x];
      if (ww != 0.0) w /= ww;
      weights[(size_t)xx * ksize + x] = w < 0 ? (int)(-0.5 + w * (1 << kResizeBits)) : (int)(0.5 + w * (1 << kResizeBits));
    }
    bounds[2 * xx] = xmin;
    bounds[2 * xx + 1] = xmax;
  }
  return ksize;
}

namespace {
struct TableEntry {
  ResizeTable t;
  std::vector<int> host;   // source of the asynchronous upload, kept alive with the entry
};
std::mutex g_tables_mu;
std::map<std::array<int, 3>, TableEntry> g_tables;   // (device, in, out)
}  // namespace

int resize_table(int in, int out, cudaStream_t s, ResizeTable* t) {
  int dev = -1;
  SE_CUDA_OK(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lk(g_tables_mu);
  auto it = g_tables.find({dev, in, out});
  if (it == g_tables.end()) {
    std::vector<int> bounds, weights;
    const int ksize = resize_coeffs(in, out, bounds, weights);
    TableEntry e;
    e.host = bounds;
    e.host.insert(e.host.end(), weights.begin(), weights.end());
    int* d = nullptr;
    SE_CUDA_OK(cudaMalloc(&d, e.host.size() * sizeof(int)));
    const cudaError_t ce = cudaMemcpyAsync(d, e.host.data(), e.host.size() * sizeof(int), cudaMemcpyHostToDevice, s);
    if (ce != cudaSuccess) cudaFree(d);
    SE_CUDA_OK(ce);
    e.t = ResizeTable{d, d + bounds.size(), ksize};
    it = g_tables.emplace(std::array<int, 3>{dev, in, out}, std::move(e)).first;
  }
  *t = it->second.t;
  return 0;
}

// One thread per output pixel, all C channels; blockIdx.y = job. Fixed-point accumulation exactly as Pillow: int32 from 2^21,
// source byte times weight, then acc >> 22 clamped to [0, 255].
template <int C, bool VERT>
__global__ void __launch_bounds__(256) resize_pass_kernel(const ResizeJob* __restrict__ jobs) {
  const ResizeJob j = jobs[blockIdx.y];
  const long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (p >= (long long)j.out_h * j.out_w) return;
  const int y = (int)(p / j.out_w), x = (int)(p - (long long)y * j.out_w);
  int v[C];
  if (j.weights == nullptr) {
    const unsigned char* s = j.in + ((size_t)y * j.in_w + x) * C;
#pragma unroll
    for (int c = 0; c < C; ++c) v[c] = s[c];
  } else {
    const int i = VERT ? y : x;
    const int lo = j.bounds[2 * i], n = j.bounds[2 * i + 1];
    const int* __restrict__ k = j.weights + (size_t)i * j.ksize;
    const size_t step = VERT ? (size_t)j.in_w * C : (size_t)C;
    const unsigned char* s = VERT ? j.in + ((size_t)lo * j.in_w + x) * C : j.in + ((size_t)y * j.in_w + lo) * C;
    int acc[C];
#pragma unroll
    for (int c = 0; c < C; ++c) acc[c] = 1 << (kResizeBits - 1);
    for (int t = 0; t < n; ++t, s += step) {
      const int w = k[t];
#pragma unroll
      for (int c = 0; c < C; ++c) acc[c] += (int)s[c] * w;
    }
#pragma unroll
    for (int c = 0; c < C; ++c) v[c] = min(max(acc[c] >> kResizeBits, 0), 255);
  }
  unsigned char* o = j.out + (size_t)p * C;
  if (j.reverse) {
#pragma unroll
    for (int c = 0; c < C; ++c) o[c] = (unsigned char)v[C - 1 - c];
  } else {
#pragma unroll
    for (int c = 0; c < C; ++c) o[c] = (unsigned char)v[c];
  }
}

int resize_pass(const ResizeJob* jobs, int njobs, long long max_pix, int C, int vertical, cudaStream_t s) {
  SE_REQUIRE(C == 1 || C == 3, "C must be 1 or 3");
  if (njobs == 0 || max_pix == 0) return 0;
  const dim3 grid((unsigned)((max_pix + 255) / 256), (unsigned)njobs);
  if (C == 1) {
    if (vertical) resize_pass_kernel<1, true><<<grid, 256, 0, s>>>(jobs);
    else resize_pass_kernel<1, false><<<grid, 256, 0, s>>>(jobs);
  } else {
    if (vertical) resize_pass_kernel<3, true><<<grid, 256, 0, s>>>(jobs);
    else resize_pass_kernel<3, false><<<grid, 256, 0, s>>>(jobs);
  }
  SE_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // namespace se
