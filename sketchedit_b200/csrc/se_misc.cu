// Glue kernels of the generator forward: input packing, heads (12->3 / 12->1 conv + tanh/sigmoid +
// blends), global pooling, mask pooling, contextual-attention operand packing and softmax, layout
// conversion. All activations are NHWC; T is the activation storage type (bf16 fast path / fp32 exact).
#include "se_common.cuh"
#include "se_misc.h"

namespace se {

template <typename T> __device__ __forceinline__ float to_f(T v);
template <> __device__ __forceinline__ float to_f<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f(float v);
template <> __device__ __forceinline__ float from_f<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f<__nv_bfloat16>(float v) { return __float2bfloat16(v); }

#define SE_DISPATCH_T(dt, ...)                          \
  if ((dt) == DT_F32) { using T = float; __VA_ARGS__; } \
  else { using T = __nv_bfloat16; __VA_ARGS__; }

static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

// ------------------------------------------------------------------------------------------ pack8
// reference editline2_g.py:62 (cat[image, sketch]) and editline_g.py:120-135 (mask-mul + cat).
template <typename T>
__global__ void pack8_kernel(const float* __restrict__ img, const float* __restrict__ sketch, const float* __restrict__ mask,
                             T* __restrict__ out, int B, int H, int W, int Wp, int padl, int img_mode, float sketch_scale,
                             int write_mask, int img2_mode) {
  // one thread per pixel of the PADDED row (Wp pixels, image at [padl, padl+W)); pads are written as zeros
  const long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const long long HW = (long long)H * W;
  if (j >= (long long)B * H * Wp) return;
  const int xp = (int)(j % Wp);
  const long long by = j / Wp;
  const int x = xp - padl;
  if (x < 0 || x >= W) {
    if (sizeof(T) == 2) {
      *reinterpret_cast<uint4*>(out + j * 8) = make_uint4(0, 0, 0, 0);
    } else {
#pragma unroll
      for (int c = 0; c < 8; ++c) out[j * 8 + c] = from_f<T>(0.0f);
    }
    return;
  }
  const long long b = by / H, pix = (by % H) * W + x;
  const long long i = b * HW + pix;
  const float m = mask ? mask[i] : 0.0f;
  const float a = img_mode == PACK_IMG_ONE ? 1.0f : (img_mode == PACK_IMG_ONE_MINUS_M ? 1.0f - m : m);
  __align__(16) T v[8];
#pragma unroll
  for (int c = 0; c < 3; ++c) v[c] = from_f<T>(img[(b * 3 + c) * HW + pix] * a);
  v[3] = from_f<T>((sketch ? sketch[i] : 1.0f) * sketch_scale);   // guide=None -> ones (reference editline_g.py:127-130)
  v[4] = from_f<T>(write_mask ? m : 0.0f);
  if (img2_mode >= 0) {   // second masked copy of the image in channels 5..7 (the style encoder's input, stem pair conv1 + wconv1)
    const float a2 = img2_mode == PACK_IMG_ONE ? 1.0f : (img2_mode == PACK_IMG_ONE_MINUS_M ? 1.0f - m : m);
#pragma unroll
    for (int c = 0; c < 3; ++c) v[5 + c] = from_f<T>(img[(b * 3 + c) * HW + pix] * a2);
  } else {
    v[5] = v[6] = v[7] = from_f<T>(0.0f);
  }
  if (sizeof(T) == 2) {
    *reinterpret_cast<uint4*>(out + j * 8) = *reinterpret_cast<const uint4*>(v);   // 8 x bf16 = one 16 B store
  } else {
#pragma unroll
    for (int c = 0; c < 8; ++c) out[j * 8 + c] = v[c];
  }
}

int pack8(const float* img, const float* sketch, const float* mask, void* out, int dt, int B, int H, int W, int Wp, int padl,
          int img_mode, float sketch_scale, int write_mask, cudaStream_t s, int img2_mode) {
  const long long n = (long long)B * H * Wp;
  SE_DISPATCH_T(dt, (pack8_kernel<T><<<cdiv(n, 256), 256, 0, s>>>(img, sketch, mask, (T*)out, B, H, W, Wp, padl, img_mode, sketch_scale, write_mask, img2_mode)));
  SE_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------ heads
// 3x3 / pad 1 conv over a 12-channel NHWC map to COUT in {1,3} channels (reference conv17 /
// conv_mask_17 / allconv17: raw conv, utils.py:27) fused with the caller-side nonlinearity:
//   HEAD_MASK   sigmoid -> soft mask (NCHW) + binarised mask plane   (editline2_g.py:93, editline2_model.py:347)
//   HEAD_TANH   tanh -> NCHW                                         (editline2_g.py:84)
//   HEAD_COARSE tanh -> [optional NCHW], xnow = t*m + img*(1-m)*(1-m) packed to 8 ch   (editline_g.py:176-181)
//   HEAD_FINE   tanh -> [optional NCHW], composed = t*soft + img*(1-soft) (NCHW)       (editline_g.py:220, editline2_model.py:132)
template <typename T, int COUT>
__global__ void head_kernel(const T* __restrict__ x, const float* __restrict__ w /*[9][12][COUT]*/, const float* __restrict__ bias,
                            int B, int H, int W, int mode, const float* __restrict__ img, const float* __restrict__ mask_bin,
                            const float* __restrict__ mask_soft, float* __restrict__ out_nchw, float* __restrict__ out2,
                            T* __restrict__ out_pack8, int no_mask_coarse, int Wp, int padl, int in_c8, long long obs, long long msbs,
                            unsigned char* __restrict__ out_u8) {
  // obs: elements between images of out_nchw (COUT*HW when dense; 4*HW when it is a view into a packed [B,4,H,W] output);
  // msbs: likewise for mask_soft
  __shared__ float ws[9 * 12 * COUT + COUT];
  for (int i = threadIdx.x; i < 9 * 12 * COUT; i += blockDim.x) ws[i] = w[i];
  if (threadIdx.x < COUT) ws[9 * 12 * COUT + threadIdx.x] = bias[threadIdx.x];
  __syncthreads();
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const long long HW = (long long)H * W;
  if (i >= B * HW) return;
  const long long b = i / HW, pix = i % HW;
  const int yy = (int)(pix / W), xx = (int)(pix % W);
  float acc[COUT];
#pragma unroll
  for (int o = 0; o < COUT; ++o) acc[o] = ws[9 * 12 * COUT + o];
#pragma unroll
  for (int t = 0; t < 9; ++t) {
    const int iy = yy + t / 3 - 1, ix = xx + t % 3 - 1;
    if (iy < 0 || iy >= H || ix < 0 || ix >= W) continue;
    // NHWC: 12 contiguous channels; C8: two channel blocks [b][2][H][W][8] (channels 12..15 are padding)
    const T* xp = in_c8 ? x + (((b * 2) * H + iy) * W + ix) * 8 : x + ((b * H + iy) * W + ix) * 12;
    const long long blk = in_c8 ? (long long)H * W * 8 - 8 : 0;
    __align__(16) T xl[16];
    if (in_c8 && sizeof(T) == 2) {   // two 16 B loads instead of twelve 2 B loads
      *reinterpret_cast<uint4*>(xl) = *reinterpret_cast<const uint4*>(xp);
      *reinterpret_cast<uint4*>(xl + 8) = *reinterpret_cast<const uint4*>(xp + blk + 8);
    } else {
#pragma unroll
      for (int c = 0; c < 12; ++c) xl[c] = xp[c + (c >= 8 ? blk : 0)];
    }
#pragma unroll
    for (int c = 0; c < 12; ++c) {
      const float xv = to_f<T>(xl[c]);
#pragma unroll
      for (int o = 0; o < COUT; ++o) acc[o] = fmaf(xv, ws[(t * 12 + c) * COUT + o], acc[o]);
    }
  }
  if (mode == HEAD_MASK) {
    const float s = 1.0f / (1.0f + expf(-acc[0]));
    out_nchw[b * obs + pix] = s;
    out2[i] = s > 0.5f ? 1.0f : 0.0f;
    if (out_u8) out_u8[i] = (unsigned char)(int)(s * 255.0f);   // test.py:25: (mask * 255).astype(uint8)
    return;
  }
  float t3[COUT];
#pragma unroll
  for (int o = 0; o < COUT; ++o) t3[o] = tanhf(acc[o]);
  if (mode == HEAD_TANH) {
#pragma unroll
    for (int o = 0; o < COUT; ++o) out_nchw[b * obs + o * HW + pix] = t3[o];
  } else if (mode == HEAD_COARSE) {
    const float m = mask_bin[i];
#pragma unroll
    for (int o = 0; o < COUT; ++o) {
      if (out_nchw) out_nchw[b * obs + o * HW + pix] = t3[o];
      const float xin = img[(b * 3 + o) * HW + pix] * (1.0f - m);
      const float v = no_mask_coarse ? t3[o] : (t3[o] * m + xin * (1.0f - m));
      out_pack8[((b * H + yy) * Wp + xx + padl) * 8 + o] = from_f<T>(v);
    }
#pragma unroll
    for (int o = COUT; o < 8; ++o) out_pack8[((b * H + yy) * Wp + xx + padl) * 8 + o] = from_f<T>(0.0f);
  } else {  // HEAD_FINE
    const float m = mask_soft[b * msbs + pix];
#pragma unroll
    for (int o = 0; o < COUT; ++o) {
      if (out2) out2[(b * COUT + o) * HW + pix] = t3[o];
      const float cv = t3[o] * m + img[(b * 3 + o) * HW + pix] * (1.0f - m);
      if (out_nchw) out_nchw[b * obs + o * HW + pix] = cv;
      if (out_u8) out_u8[i * 3 + (2 - o)] = (unsigned char)(int)((cv + 1.0f) / 2.0f * 255.0f);   // test.py:26-35: truncate, HWC, RGB -> BGR
    }
  }
}

// bf16 channel-blocked input (the tensor-core path): same arithmetic, organised for the FP32 pipe.
//   * weights come in as a by-value kernel parameter: they sit in the constant bank and feed the FMAs directly
//     (the generic kernel spends one shared-memory load per FMA)
//   * channels are processed in pairs with the packed fma.rn.f32x2 (two FMAs per issue slot): a bf16x2 word expands
//     to the (even, odd) channel pair, the weights are stored as matching pairs, and each output keeps an (even, odd)
//     pair of partial sums that is added at the end
template <int COUT>
struct HeadWeights {
  float2 w[9][6][COUT];   // [tap][channel pair][out] = (w[tap][2p][o], w[tap][2p+1][o])
  float b[COUT];
};
__device__ __forceinline__ unsigned long long ffma2(unsigned long long a, unsigned long long b, unsigned long long c) {
  unsigned long long d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
template <int COUT>
__global__ void __launch_bounds__(128) head_c8_kernel(const __nv_bfloat16* __restrict__ x, const __grid_constant__ HeadWeights<COUT> hw, int B, int H,
                                                      int W, int mode, const float* __restrict__ img, const float* __restrict__ mask_bin,
                                                      const float* __restrict__ mask_soft, float* __restrict__ out_nchw,
                                                      float* __restrict__ out2, __nv_bfloat16* __restrict__ out_pack8, int no_mask_coarse,
                                                      int Wp, int padl, long long obs, long long msbs, unsigned char* __restrict__ out_u8) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const long long HW = (long long)H * W;
  if (i >= B * HW) return;
  const long long b = i / HW, pix = i % HW;
  const int yy = (int)(pix / W), xx = (int)(pix % W);
  unsigned long long acc[COUT];
#pragma unroll
  for (int o = 0; o < COUT; ++o) acc[o] = 0ull;
  const uint4* plane0 = reinterpret_cast<const uint4*>(x) + (b * 2) * HW;   // [b][2 blocks][H][W] x 16 B
#pragma unroll
  for (int t = 0; t < 9; ++t) {
    const int iy = yy + t / 3 - 1, ix = xx + t % 3 - 1;
    if (iy < 0 || iy >= H || ix < 0 || ix >= W) continue;
    const uint4 q0 = plane0[(long long)iy * W + ix];
    const uint4 q1 = plane0[HW + (long long)iy * W + ix];             // channels 8..15 (12..15 are padding)
    const uint32_t wds[6] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y};
#pragma unroll
    for (int p = 0; p < 6; ++p) {
      // bf16x2 -> (even channel, odd channel) as an fp32 pair
      const unsigned long long xp = ((unsigned long long)(wds[p] & 0xffff0000u) << 32) | (unsigned long long)(wds[p] << 16);
#pragma unroll
      for (int o = 0; o < COUT; ++o) {
        const float2 wv = hw.w[t][p][o];
        const unsigned long long wp = ((unsigned long long)__float_as_uint(wv.y) << 32) | __float_as_uint(wv.x);
        acc[o] = ffma2(xp, wp, acc[o]);
      }
    }
  }
  float r[COUT];
#pragma unroll
  for (int o = 0; o < COUT; ++o) r[o] = hw.b[o] + (__uint_as_float((uint32_t)acc[o]) + __uint_as_float((uint32_t)(acc[o] >> 32)));
  if (mode == HEAD_MASK) {
    const float sg = 1.0f / (1.0f + expf(-r[0]));
    out_nchw[b * obs + pix] = sg;
    out2[i] = sg > 0.5f ? 1.0f : 0.0f;
    if (out_u8) out_u8[i] = (unsigned char)(int)(sg * 255.0f);   // test.py:25: (mask * 255).astype(uint8)
    return;
  }
  float t3[COUT];
#pragma unroll
  for (int o = 0; o < COUT; ++o) t3[o] = tanhf(r[o]);
  if (mode == HEAD_TANH) {
#pragma unroll
    for (int o = 0; o < COUT; ++o) out_nchw[b * obs + o * HW + pix] = t3[o];
  } else if (mode == HEAD_COARSE) {
    const float m = mask_bin[i];
    __align__(16) __nv_bfloat16 pk[8];
#pragma unroll
    for (int o = 0; o < 8; ++o) pk[o] = __float2bfloat16(0.0f);
#pragma unroll
    for (int o = 0; o < COUT; ++o) {
      if (out_nchw) out_nchw[b * obs + o * HW + pix] = t3[o];
      const float xin = img[(b * 3 + o) * HW + pix] * (1.0f - m);
      pk[o] = __float2bfloat16(no_mask_coarse ? t3[o] : (t3[o] * m + xin * (1.0f - m)));
    }
    *reinterpret_cast<uint4*>(out_pack8 + ((b * H + yy) * Wp + xx + padl) * 8) = *reinterpret_cast<const uint4*>(pk);
  } else {  // HEAD_FINE
    const float m = mask_soft[b * msbs + pix];
#pragma unroll
    for (int o = 0; o < COUT; ++o) {
      if (out2) out2[(b * COUT + o) * HW + pix] = t3[o];
      const float cv = t3[o] * m + img[(b * 3 + o) * HW + pix] * (1.0f - m);
      if (out_nchw) out_nchw[b * obs + o * HW + pix] = cv;
      if (out_u8) out_u8[i * 3 + (2 - o)] = (unsigned char)(int)((cv + 1.0f) / 2.0f * 255.0f);   // test.py:26-35: truncate, HWC, RGB -> BGR
    }
  }
}

template <int COUT>
static int head_c8_launch(const void* x, const float* w_host, const float* b_host, int B, int H, int W, int mode, const float* img,
                          const float* mask_bin, const float* mask_soft, float* out_nchw, float* out2, void* out_pack8, int no_mask_coarse,
                          int Wp, int padl, long long obs, long long msbs, unsigned char* out_u8, cudaStream_t s) {
  HeadWeights<COUT> hw;
  for (int t = 0; t < 9; ++t)
    for (int p = 0; p < 6; ++p)
      for (int o = 0; o < COUT; ++o) hw.w[t][p][o] = make_float2(w_host[(t * 12 + 2 * p) * COUT + o], w_host[(t * 12 + 2 * p + 1) * COUT + o]);
  for (int o = 0; o < COUT; ++o) hw.b[o] = b_host[o];
  const long long n = (long long)B * H * W;
  head_c8_kernel<COUT><<<cdiv(n, 128), 128, 0, s>>>((const __nv_bfloat16*)x, hw, B, H, W, mode, img, mask_bin, mask_soft, out_nchw, out2,
                                                    (__nv_bfloat16*)out_pack8, no_mask_coarse, Wp, padl, obs ? obs : (long long)COUT * H * W,
                                                    msbs ? msbs : (long long)H * W, out_u8);
  SE_CUDA_OK(cudaGetLastError());
  return 0;
}
// w_host / b_host: host copies of the [9][12][cout] weights and the bias (kernel parameters are built from them)
int head_c8(const void* x, const float* w_host, const float* b_host, int cout, int B, int H, int W, int mode, const float* img,
            const float* mask_bin, const float* mask_soft, float* out_nchw, float* out2, void* out_pack8, int no_mask_coarse, int Wp, int padl,
            long long obs, long long msbs, unsigned char* out_u8, cudaStream_t s) {
  SE_REQUIRE(cout == 1 || cout == 3, "head cout");
  if (cout == 1) return head_c8_launch<1>(x, w_host, b_host, B, H, W, mode, img, mask_bin, mask_soft, out_nchw, out2, out_pack8, no_mask_coarse, Wp, padl, obs, msbs, out_u8, s);
  return head_c8_launch<3>(x, w_host, b_host, B, H, W, mode, img, mask_bin, mask_soft, out_nchw, out2, out_pack8, no_mask_coarse, Wp, padl, obs, msbs, out_u8, s);
}

int head(const void* x, int dt, int in_c8, const float* w, const float* bias, int cout, int B, int H, int W, int mode, const float* img,
         const float* mask_bin, const float* mask_soft, float* out_nchw, float* out2, void* out_pack8, int no_mask_coarse,
         int Wp, int padl, long long obs, long long msbs, unsigned char* out_u8, cudaStream_t s) {
  const long long n = (long long)B * H * W;
  SE_REQUIRE(cout == 1 || cout == 3, "head cout");
  if (!obs) obs = (long long)cout * H * W;
  if (!msbs) msbs = (long long)H * W;
  SE_DISPATCH_T(dt, {
    if (cout == 1)
      head_kernel<T, 1><<<cdiv(n, 128), 128, 0, s>>>((const T*)x, w, bias, B, H, W, mode, img, mask_bin, mask_soft, out_nchw, out2, (T*)out_pack8, no_mask_coarse, Wp, padl, in_c8, obs, msbs, out_u8);
    else
      head_kernel<T, 3><<<cdiv(n, 128), 128, 0, s>>>((const T*)x, w, bias, B, H, W, mode, img, mask_bin, mask_soft, out_nchw, out2, (T*)out_pack8, no_mask_coarse, Wp, padl, in_c8, obs, msbs, out_u8);
  });
  SE_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------ plane reductions
// per (image, channel) reduction over the h x w plane of an NHWC map:
//   RED_MAX / RED_AVG      global pooling            (editline_g.py:160-165)
//   RED_RNORM              1/sqrt(sum x^2 + 1e-8)    (splitcam.py:40)
template <typename T>
__global__ void plane_reduce_kernel(const T* __restrict__ x, int ldx, int c8, int C, int HW, int mode, float* __restrict__ out) {
  __shared__ float red[8][33];
  const int b = blockIdx.y;
  const int c = blockIdx.x * 32 + threadIdx.x;
  float acc = (mode == RED_MAX) ? -INFINITY : 0.0f;
  if (c < C) {
    // NHWC: pixel pitch ldx; C8: [b][ldx blocks][HW][8]
    const T* xp = c8 ? x + ((size_t)b * ldx + (c >> 3)) * HW * 8 + (c & 7) : x + (size_t)b * HW * ldx + c;
    const size_t pitch = c8 ? 8 : ldx;
    for (int p = threadIdx.y; p < HW; p += 8) {
      const float v = to_f<T>(xp[(size_t)p * pitch]);
      if (mode == RED_MAX) acc = fmaxf(acc, v);
      else if (mode == RED_AVG) acc += v;
      else acc = fmaf(v, v, acc);
    }
  }
  red[threadIdx.y][threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.y == 0 && c < C) {
    for (int j = 1; j < 8; ++j) {
      const float v = red[j][threadIdx.x];
      acc = (mode == RED_MAX) ? fmaxf(acc, v) : acc + v;
    }
    if (mode == RED_AVG) acc /= (float)HW;
    if (mode == RED_RNORM) acc = 1.0f / sqrtf(acc + 1e-8f);
    out[(size_t)b * C + c] = acc;
  }
}

// C8 bf16: one block per (image, channel block): the plane is HW contiguous 16 B pixels
__global__ void plane_reduce_c8_kernel(const __nv_bfloat16* __restrict__ x, int ldx, int C, int HW, int mode, float* __restrict__ out) {
  __shared__ float red[8][8];
  const int b = blockIdx.y, cb = blockIdx.x;
  const uint4* xp = reinterpret_cast<const uint4*>(x + ((size_t)b * ldx + cb) * HW * 8);
  float acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = (mode == RED_MAX) ? -INFINITY : 0.0f;
  for (int p = threadIdx.x; p < HW; p += blockDim.x) {
    const uint4 q = xp[p];
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&q);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 v = __bfloat1622float2(h[i]);
      if (mode == RED_MAX) { acc[2 * i] = fmaxf(acc[2 * i], v.x); acc[2 * i + 1] = fmaxf(acc[2 * i + 1], v.y); }
      else if (mode == RED_AVG) { acc[2 * i] += v.x; acc[2 * i + 1] += v.y; }
      else { acc[2 * i] = fmaf(v.x, v.x, acc[2 * i]); acc[2 * i + 1] = fmaf(v.y, v.y, acc[2 * i + 1]); }
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i)
    for (int o = 16; o; o >>= 1) {
      const float t = __shfl_xor_sync(0xffffffffu, acc[i], o);
      acc[i] = (mode == RED_MAX) ? fmaxf(acc[i], t) : acc[i] + t;
    }
  const int wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  if ((threadIdx.x & 31) == 0)
    for (int i = 0; i < 8; ++i) red[wid][i] = acc[i];
  __syncthreads();
  if (threadIdx.x < 8) {
    float r = red[0][threadIdx.x];
    for (int j = 1; j < nw; ++j) r = (mode == RED_MAX) ? fmaxf(r, red[j][threadIdx.x]) : r + red[j][threadIdx.x];
    if (mode == RED_AVG) r /= (float)HW;
    if (mode == RED_RNORM) r = 1.0f / sqrtf(r + 1e-8f);
    const int c = cb * 8 + threadIdx.x;
    if (c < C) out[(size_t)b * C + c] = r;
  }
}

// NHWC bf16 with C % 8 == 0: blocks over (pixel slices, image); partial results combined with float atomics
// (max: order-free; sums: used for the L2 norm only where the bf16 path tolerates re-association)
// NHWC bf16 sum-of-squares over slices of the plane: partial sums combined with atomicAdd (used for the attention
// key norm only; re-association is far below bf16 resolution), then 1/sqrt(sum + 1e-8)
__global__ void plane_sumsq_nhwc_kernel(const __nv_bfloat16* __restrict__ x, int ldx, int C, int HW, int slices, float* __restrict__ acc) {
  __shared__ float red[8][33];
  const int b = blockIdx.y, sl = blockIdx.z;
  const int c = blockIdx.x * 32 + threadIdx.x;
  const int p0 = (int)((long long)HW * sl / slices), p1 = (int)((long long)HW * (sl + 1) / slices);
  float a = 0.0f;
  if (c < C) {
    const __nv_bfloat16* xp = x + (size_t)b * HW * ldx + c;
    for (int p = p0 + threadIdx.y; p < p1; p += 8) {
      const float v = __bfloat162float(xp[(size_t)p * ldx]);
      a = fmaf(v, v, a);
    }
  }
  red[threadIdx.y][threadIdx.x] = a;
  __syncthreads();
  if (threadIdx.y == 0 && c < C) {
    for (int j = 1; j < 8; ++j) a += red[j][threadIdx.x];
    atomicAdd(acc + (size_t)b * C + c, a);
  }
}
__global__ void rnorm_finalize_kernel(float* __restrict__ v, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) v[i] = 1.0f / sqrtf(v[i] + 1e-8f);
}

int plane_reduce(const void* x, int dt, int B, int HW, int C, int ldx, int c8, int mode, float* out, cudaStream_t s) {
  if (!c8 && dt == DT_BF16 && mode == RED_RNORM && HW >= 1024) {
    const int slices = 16;
    SE_CUDA_OK(cudaMemsetAsync(out, 0, (size_t)B * C * 4, s));
    dim3 grid(cdiv(C, 32), B, slices), block(32, 8);
    plane_sumsq_nhwc_kernel<<<grid, block, 0, s>>>((const __nv_bfloat16*)x, ldx, C, HW, slices, out);
    rnorm_finalize_kernel<<<cdiv((long long)B * C, 256), 256, 0, s>>>(out, B * C);
    SE_CUDA_OK(cudaGetLastError());
    return 0;
  }
  if (c8 && dt == DT_BF16) {
    dim3 grid((C + 7) / 8, B);
    plane_reduce_c8_kernel<<<grid, 256, 0, s>>>((const __nv_bfloat16*)x, ldx, C, HW, mode, out);
    SE_CUDA_OK(cudaGetLastError());
    return 0;
  }
  dim3 grid(cdiv(C, 32), B), block(32, 8);
  SE_DISPATCH_T(dt, (plane_reduce_kernel<T><<<grid, block, 0, s>>>((const T*)x, ldx, c8, C, HW, mode, out)));
  SE_CUDA_OK(cudaGetLastError());
  return 0;
}

// nearest 1x1 -> h x w broadcast of the pooled vector into channels [choff, choff+C) of an NHWC map
// (editline_g.py:166-167: interpolate + cat).
template <typename T>
__global__ void broadcast_kernel(const float* __restrict__ v, T* __restrict__ y, int C, int HW, int ldo, int choff, int c8, long long total) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= total) return;
  if (c8) {   // [b][ldo blocks][HW][8]: i enumerates (b, c/8, p, c%8) so that consecutive threads write consecutive bytes
    const int c7 = (int)(i & 7);
    long long r = i >> 3;
    const long long p = r % HW; r /= HW;
    const int cb = (int)(r % (C >> 3));
    const long long b = r / (C >> 3);
    y[((b * ldo + (choff >> 3) + cb) * HW + p) * 8 + c7] = from_f<T>(v[b * C + cb * 8 + c7]);
    return;
  }
  const int c = (int)(i % C);
  const long long pix = i / C;
  const long long b = pix / HW;
  y[pix * ldo + choff + c] = from_f<T>(v[b * C + c]);
}

__global__ void broadcast_c8_kernel(const float* __restrict__ v, __nv_bfloat16* __restrict__ y, int C, int HW, int ldo, int choff, long long total) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;   // (b, cb, p)
  if (i >= total) return;
  const long long p = i % HW;
  long long r = i / HW;
  const int cb = (int)(r % (C >> 3));
  const long long b = r / (C >> 3);
  const float* src = v + b * C + cb * 8;
  const uint4 q = make_uint4(pack_bf16x2(src[0], src[1]), pack_bf16x2(src[2], src[3]), pack_bf16x2(src[4], src[5]), pack_bf16x2(src[6], src[7]));
  *reinterpret_cast<uint4*>(y + ((b * ldo + (choff >> 3) + cb) * HW + p) * 8) = q;
}

int broadcast_channels(const float* v, void* y, int dt, int B, int HW, int C, int ldo, int choff, int c8, cudaStream_t s) {
  if (c8 && dt == DT_BF16 && C % 8 == 0 && choff % 8 == 0) {
    const long long n = (long long)B * (C >> 3) * HW;
    broadcast_c8_kernel<<<cdiv(n, 256), 256, 0, s>>>(v, (__nv_bfloat16*)y, C, HW, ldo, choff, n);
    SE_CUDA_OK(cudaGetLastError());
    return 0;
  }
  const long long total = (long long)B * HW * C;
  SE_REQUIRE(!c8 || (C % 8 == 0 && choff % 8 == 0), "C8 broadcast needs whole channel blocks");
  SE_DISPATCH_T(dt, (broadcast_kernel<T><<<cdiv(total, 256), 256, 0, s>>>(v, (T*)y, C, HW, ldo, choff, c8, total)));
  SE_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------ mask pooling
// avg_pool2d(mask, 4, 4) (editline_g.py:204) and the per-key valid flag of cam_1
// (splitcam.py:49-53,89-90: mean over the 4x4 patch of (1 - mask_s) > th).
__global__ void avgpool4_kernel(const float* __restrict__ m, float* __restrict__ out, int B, int H, int W) {
  const int h = H / 4, w = W / 4;
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= (long long)B * h * w) return;
  const int x = (int)(i % w), y = (int)((i / w) % h);
  const long long b = i / ((long long)h * w);
  float a = 0.0f;
  for (int u = 0; u < 4; ++u)
    for (int v = 0; v < 4; ++v) a += m[(b * H + 4 * y + u) * W + 4 * x + v];
  out[i] = a * (1.0f / 16.0f);
}

int avgpool4(const float* m, float* out, int B, int H, int W, cudaStream_t s) {
  avgpool4_kernel<<<cdiv((long long)B * (H / 4) * (W / 4), 256), 256, 0, s>>>(m, out, B, H, W);
  SE_CUDA_OK(cudaGetLastError());
  return 0;
}

__global__ void cam_colmask_kernel(const float* __restrict__ mask_s, float* __restrict__ out, int B, int h, int w, int hs, int ws,
                                   int patch, int stride, float th) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= (long long)B * hs * ws) return;
  const int lx = (int)(i % ws), ly = (int)((i / ws) % hs);
  const long long b = i / ((long long)hs * ws);
  float a = 0.0f;
  for (int u = 0; u < patch; ++u)
    for (int v = 0; v < patch; ++v) a += 1.0f - mask_s[(b * h + ly * stride + u) * w + lx * stride + v];
  // the reference takes mean over v then over u of exact multiples of 1/16: the order does not matter
  out[i] = (a / (float)(patch * patch) > th) ? 1.0f : 0.0f;
}

int cam_colmask(const float* mask_s, float* out, int B, int h, int w, int hs, int ws, float th, cudaStream_t s) {
  cam_colmask_kernel<<<cdiv((long long)B * hs * ws, 256), 256, 0, s>>>(mask_s, out, B, h, w, hs, ws, 4, 2, th);
  SE_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------ attention operands
// Keys  K[l][(u,v,c)] = f[2ly+u, 2lx+v, c] * rnorm[c]        (splitcam.py:39-44, norm_type 1, 4x4 / stride 2)
// direct layout: fp32 [b][tap][c][CoutP]
template <typename T>
__global__ void cam_pack_k_direct_kernel(const T* __restrict__ f, const float* __restrict__ rnorm, float* __restrict__ out,
                                         int B, int h, int w, int C, int ws, int L, int CoutP, long long total) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int l = (int)(i % CoutP);
  long long r = i / CoutP;
  const int c = (int)(r % C); r /= C;
  const int tap = (int)(r % 16);
  const long long b = r / 16;
  float v = 0.0f;
  if (l < L) {
    const int ly = l / ws, lx = l % ws, u = tap / 4, vv = tap % 4;
    v = to_f<T>(f[((b * h + 2 * ly + u) * w + 2 * lx + vv) * C + c]) * rnorm[b * C + c];
  }
  out[i] = v;
}

int cam_pack_k(const void* f, int dt, const float* rnorm, void* out, int B, int h, int w, int C, int ws, int L, int Lpad, cudaStream_t s) {
  const long long total = (long long)B * 16 * C * Lpad;
  SE_DISPATCH_T(dt, (cam_pack_k_direct_kernel<T><<<cdiv(total, 256), 256, 0, s>>>((const T*)f, rnorm, (float*)out, B, h, w, C, ws, L, Lpad, total)));
  SE_CUDA_OK(cudaGetLastError());
  return 0;
}

// Values for the fold-sum written as 4 sub-pixel (parity) 2x2 "convolutions" over the token image
// P[b, ny, nx, l] (splitcam.py:152, utils.py:102-128):
//   out[2yy+py, 2xx+px, c] = sum_{a,b in {0,1}} sum_l P[yy-a, xx-b, l] * f[2ly+py+2a, 2lx+px+2b, c]
// direct layout: fp32 [pc][b][tap][l (Ci = Lpad)][CoutP = C]
template <typename T>
__global__ void cam_pack_v_direct_kernel(const T* __restrict__ f, float* __restrict__ out, int B, int h, int w, int C, int ws, int L,
                                         int Lpad, long long total) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int c = (int)(i % C);
  long long r = i / C;
  const int l = (int)(r % Lpad); r /= Lpad;
  const int tap = (int)(r % 4); r /= 4;
  const long long b = r % B;
  const int pc = (int)(r / B);
  float v = 0.0f;
  if (l < L) {
    const int ly = l / ws, lx = l % ws, py = pc / 2, px = pc % 2, a = tap / 2, bb = tap % 2;
    v = to_f<T>(f[((b * h + 2 * ly + py + 2 * a) * w + 2 * lx + px + 2 * bb) * C + c]);
  }
  out[i] = v;
}

int cam_pack_v(const void* f, int dt, void* out, int B, int h, int w, int C, int ws, int L, int Lpad, cudaStream_t s) {
  const long long total = 4LL * B * 4 * Lpad * C;
  SE_DISPATCH_T(dt, (cam_pack_v_direct_kernel<T><<<cdiv(total, 256), 256, 0, s>>>((const T*)f, (float*)out, B, h, w, C, ws, L, Lpad, total)));
  SE_CUDA_OK(cudaGetLastError());
  return 0;
}

// softmax over the key axis of the logits S[row][0..L) (fp32, row pitch lds) -> P[row][0..Lpad) with
// zero padding (splitcam.py:105; the scale 10 and the key mask are already applied by the GEMM epilogue).
template <typename T>
__global__ void softmax_rows_kernel(const float* __restrict__ S, int lds, T* __restrict__ P, int ldp, int L) {
  // one 256-thread block per row; up to SM_MAXV values per thread stay in registers (rows <= 256*SM_MAXV keys),
  // longer rows fall back to re-reading
  constexpr int SM_MAXV = 16;
  __shared__ float red[32];
  const long long row = blockIdx.x;
  const float* s = S + row * lds;
  T* p = P + row * ldp;
  const bool fits = L <= 256 * SM_MAXV;
  float v[SM_MAXV];
  float mx = -INFINITY;
#pragma unroll
  for (int k = 0; k < SM_MAXV; ++k) {
    const int i = threadIdx.x + k * 256;
    v[k] = (fits && i < L) ? s[i] : -INFINITY;
    mx = fmaxf(mx, v[k]);
  }
  if (!fits)
    for (int i = threadIdx.x; i < L; i += 256) mx = fmaxf(mx, s[i]);
  for (int o = 16; o; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
  __syncthreads();
  mx = red[0];
  for (int i = 1; i < 8; ++i) mx = fmaxf(mx, red[i]);
  __syncthreads();
  float sum = 0.0f;
  if (fits) {
#pragma unroll
    for (int k = 0; k < SM_MAXV; ++k) {
      v[k] = expf(v[k] - mx);      // exp(-inf) = 0 for the padding lanes
      sum += v[k];
    }
  } else {
    for (int i = threadIdx.x; i < L; i += 256) sum += expf(s[i] - mx);
  }
  for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = sum;
  __syncthreads();
  sum = 0.0f;
  for (int i = 0; i < 8; ++i) sum += red[i];
  const float inv = 1.0f / sum;
  if (fits) {
#pragma unroll
    for (int k = 0; k < SM_MAXV; ++k) {
      const int i = threadIdx.x + k * 256;
      if (i < ldp) p[i] = from_f<T>(i < L ? v[k] * inv : 0.0f);
    }
  } else {
    for (int i = threadIdx.x; i < ldp; i += 256) p[i] = from_f<T>(i < L ? expf(s[i] - mx) * inv : 0.0f);
  }
}

// rows of <= 1024 keys with 16 B aligned pitches: one WARP per row, the row lives in registers (32 values per lane,
// float4 loads), reductions are shuffles only - no block barriers, one pass over the logits
__global__ void __launch_bounds__(256) softmax_rows_warp_kernel(const float* __restrict__ S, int lds, __nv_bfloat16* __restrict__ P, int ldp, int L,
                                                                long long rows) {
  const long long row = blockIdx.x * 8LL + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const float4* s4 = reinterpret_cast<const float4*>(S + row * lds);
  float v[32];
  float mx = -INFINITY;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int i = (k * 32 + lane) * 4;
    float4 q = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    if (i < L) q = s4[k * 32 + lane];                  // i % 4 == 0 and the pitch covers the padded row
    v[4 * k] = q.x;
    v[4 * k + 1] = (i + 1 < L) ? q.y : -INFINITY;
    v[4 * k + 2] = (i + 2 < L) ? q.z : -INFINITY;
    v[4 * k + 3] = (i + 3 < L) ? q.w : -INFINITY;
    mx = fmaxf(fmaxf(mx, v[4 * k]), fmaxf(fmaxf(v[4 * k + 1], v[4 * k + 2]), v[4 * k + 3]));
  }
  for (int o = 16; o; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float sum = 0.0f;
#pragma unroll
  for (int k = 0; k < 32; ++k) {
    v[k] = expf(v[k] - mx);                             // exp(-inf) = 0 for the padding lanes
    sum += v[k];
  }
  for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  const float inv = 1.0f / sum;
  uint2* p2 = reinterpret_cast<uint2*>(P + row * ldp);
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int i = (k * 32 + lane) * 4;
    if (i < ldp) p2[k * 32 + lane] = make_uint2(pack_bf16x2(v[4 * k] * inv, v[4 * k + 1] * inv), pack_bf16x2(v[4 * k + 2] * inv, v[4 * k + 3] * inv));
  }
}

int softmax_rows(const float* S, int lds, void* P, int dt, int ldp, long long rows, int L, cudaStream_t s) {
  if (dt == DT_BF16 && L <= 1024 && lds % 4 == 0 && ldp % 4 == 0 && lds >= ((L + 3) & ~3) && ldp <= 1024 &&
      (reinterpret_cast<uintptr_t>(S) & 15) == 0 && (reinterpret_cast<uintptr_t>(P) & 7) == 0) {
    softmax_rows_warp_kernel<<<(unsigned)cdiv(rows, 8), 256, 0, s>>>(S, lds, (__nv_bfloat16*)P, ldp, L, rows);
    SE_CUDA_OK(cudaGetLastError());
    return 0;
  }
  SE_DISPATCH_T(dt, (softmax_rows_kernel<T><<<(unsigned)rows, 256, 0, s>>>(S, lds, (T*)P, ldp, L)));
  SE_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------ layout conversion
template <typename T>
__global__ void nchw_to_nhwc_kernel(const float* __restrict__ x, T* __restrict__ y, int C, int HW, int ldo, int choff, long long total) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int c = (int)(i % C);
  const long long pix = i / C;
  const long long b = pix / HW, p = pix % HW;
  y[pix * ldo + choff + c] = from_f<T>(x[(b * C + c) * HW + p]);
}
template <typename T>
__global__ void nhwc_to_nchw_kernel(const T* __restrict__ x, float* __restrict__ y, int C, int HW, int ldx, int choff, long long total) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long p = i % HW;
  const long long r = i / HW;
  const int c = (int)(r % C);
  const long long b = r / C;
  y[i] = to_f<T>(x[(b * HW + p) * ldx + choff + c]);
}

// NCHW fp32 [B,cin<=8,H,W] -> packed 8-channel rows of Wp pixels (image at [padl, padl+W)); pads/extra channels untouched
template <typename T>
__global__ void nchw_to_stem8_kernel(const float* __restrict__ x, T* __restrict__ y, int cin, int H, int W, int Wp, int padl, long long total) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int c = (int)(i % cin);
  long long r = i / cin;
  const int xx = (int)(r % W); r /= W;
  const int yy = (int)(r % H);
  const long long b = r / H;
  y[((b * H + yy) * Wp + xx + padl) * 8 + c] = from_f<T>(x[((b * cin + c) * H + yy) * W + xx]);
}
int nchw_to_stem8(const float* x, void* y, int dt, int B, int cin, int H, int W, int Wp, int padl, cudaStream_t s) {
  const long long total = (long long)B * cin * H * W;
  SE_REQUIRE(cin <= 8, "stem input channels");
  SE_DISPATCH_T(dt, (nchw_to_stem8_kernel<T><<<cdiv(total, 256), 256, 0, s>>>(x, (T*)y, cin, H, W, Wp, padl, total)));
  SE_CUDA_OK(cudaGetLastError());
  return 0;
}

// NCHW fp32 -> C8 bf16 [B][ceil(C/8)][HW][8] (padding channels untouched: zero the buffer first when C % 8)
__global__ void nchw_to_c8_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ y, int C, int HW, long long total) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long p = i % HW;
  long long r = i / HW;
  const int c = (int)(r % C);
  const long long b = r / C;
  const int CB = (C + 7) / 8;
  y[((b * CB + (c >> 3)) * HW + p) * 8 + (c & 7)] = __float2bfloat16(x[i]);
}
int nchw_to_c8(const float* x, void* y, int B, int C, int HW, cudaStream_t s) {
  const long long total = (long long)B * C * HW;
  nchw_to_c8_kernel<<<cdiv(total, 256), 256, 0, s>>>(x, (__nv_bfloat16*)y, C, HW, total);
  SE_CUDA_OK(cudaGetLastError());
  return 0;
}

// NCHW fp32 -> space-to-depth C8 bf16 [B][4*C/8][H/2][W/2][8]: pixel (y, x) channel c lands in channel block
// ((y&1)*2 + (x&1)) * C/8 + c/8 at position (y/2, x/2)  (C % 8 == 0, H and W even)
__global__ void nchw_to_c8_s2d_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ y, int C, int H, int W, long long total) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int px = (int)(i % W);
  long long r = i / W;
  const int py = (int)(r % H);
  r /= H;
  const int c = (int)(r % C);
  const long long b = r / C;
  const int CB = C / 8, Hs = H / 2, Ws = W / 2;
  const int blk = ((py & 1) * 2 + (px & 1)) * CB + (c >> 3);
  y[(((b * 4 * CB + blk) * Hs + (py >> 1)) * Ws + (px >> 1)) * 8 + (c & 7)] = __float2bfloat16(x[i]);
}
int nchw_to_c8_s2d(const float* x, void* y, int B, int C, int H, int W, cudaStream_t s) {
  SE_REQUIRE(C % 8 == 0 && H % 2 == 0 && W % 2 == 0, "space-to-depth C8 needs C % 8 == 0 and even H, W");
  const long long total = (long long)B * C * H * W;
  nchw_to_c8_s2d_kernel<<<cdiv(total, 256), 256, 0, s>>>(x, (__nv_bfloat16*)y, C, H, W, total);
  SE_CUDA_OK(cudaGetLastError());
  return 0;
}

// C8 bf16 [B][C/8][HW][8] -> NCHW fp32 (C % 8 == 0)
__global__ void c8_to_nchw_kernel(const __nv_bfloat16* __restrict__ x, float* __restrict__ y, int C, int HW, long long total) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= total) return;
  const long long p = i % HW;
  long long r = i / HW;
  const int c = (int)(r % C);
  const long long b = r / C;
  y[i] = __bfloat162float(x[((b * (C / 8) + (c >> 3)) * HW + p) * 8 + (c & 7)]);
}
int c8_to_nchw(const void* x, float* y, int B, int C, int HW, cudaStream_t s) {
  SE_REQUIRE(C % 8 == 0, "C8 -> NCHW needs whole channel blocks");
  const long long total = (long long)B * C * HW;
  c8_to_nchw_kernel<<<cdiv(total, 256), 256, 0, s>>>((const __nv_bfloat16*)x, y, C, HW, total);
  SE_CUDA_OK(cudaGetLastError());
  return 0;
}

int nchw_to_nhwc(const float* x, void* y, int dt, int B, int C, int HW, int ldo, int choff, cudaStream_t s) {
  const long long total = (long long)B * C * HW;
  SE_DISPATCH_T(dt, (nchw_to_nhwc_kernel<T><<<cdiv(total, 256), 256, 0, s>>>(x, (T*)y, C, HW, ldo, choff, total)));
  SE_CUDA_OK(cudaGetLastError());
  return 0;
}
int nhwc_to_nchw(const void* x, int dt, float* y, int B, int C, int HW, int ldx, int choff, cudaStream_t s) {
  const long long total = (long long)B * C * HW;
  SE_DISPATCH_T(dt, (nhwc_to_nchw_kernel<T><<<cdiv(total, 256), 256, 0, s>>>((const T*)x, y, C, HW, ldx, choff, total)));
  SE_CUDA_OK(cudaGetLastError());
  return 0;
}

// reference data/testimage_dataset.py:89-103 on device: image uint8 HWC RGB -> fp32 NCHW (ToTensor: /255; Normalize(0.5, 0.5)),
// sketch uint8 (already resized to the image) -> {0, 1} fp32 (ToTensor then > 0)
__global__ void u8_to_inputs_kernel(const unsigned char* __restrict__ img_u8, const unsigned char* __restrict__ sk_u8, float* __restrict__ img,
                                    float* __restrict__ sk, int B, long long HW) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= B * HW) return;
  const long long b = i / HW, pix = i % HW;
#pragma unroll
  for (int c = 0; c < 3; ++c) img[(b * 3 + c) * HW + pix] = (__fdiv_rn((float)img_u8[i * 3 + c], 255.0f) - 0.5f) / 0.5f;
  sk[i] = sk_u8[i] > 0 ? 1.0f : 0.0f;
}
int u8_to_inputs(const unsigned char* img_u8, const unsigned char* sk_u8, float* img, float* sk, int B, int H, int W, cudaStream_t s) {
  const long long HW = (long long)H * W;
  u8_to_inputs_kernel<<<cdiv(B * HW, 256), 256, 0, s>>>(img_u8, sk_u8, img, sk, B, HW);
  SE_CUDA_OK(cudaGetLastError());
  return 0;
}

// inputs of the region inpaint (reference editline2_model.py:343-345: line_inpaint = line_full * mask_inpaint): uint8 entry
// (T = unsigned char): image HWC RGB -> fp32 NCHW as u8_to_inputs_kernel, R = region > 0, s*R with s = sketch > 0; float entry
// (T = float, img_u8 and region NULL): only s*R from the caller's planes
__device__ __forceinline__ float region_plane(unsigned char v) { return v > 0 ? 1.0f : 0.0f; }
__device__ __forceinline__ float region_plane(float v) { return v; }
template <typename T>
__global__ void region_inputs_kernel(const unsigned char* __restrict__ img_u8, const T* __restrict__ sk_in, const T* __restrict__ rg_in,
                                     float* __restrict__ img, float* __restrict__ region, float* __restrict__ sk_region, int B, long long HW) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= B * HW) return;
  if (img_u8) {
    const long long b = i / HW, pix = i % HW;
#pragma unroll
    for (int c = 0; c < 3; ++c) img[(b * 3 + c) * HW + pix] = (__fdiv_rn((float)img_u8[i * 3 + c], 255.0f) - 0.5f) / 0.5f;
  }
  const float r = region_plane(rg_in[i]);
  if (region) region[i] = r;
  sk_region[i] = region_plane(sk_in[i]) * r;
}
int region_inputs_u8(const unsigned char* img_u8, const unsigned char* sk_u8, const unsigned char* rg_u8, float* img, float* region, float* sk_region,
                     int B, int H, int W, cudaStream_t s) {
  const long long HW = (long long)H * W;
  region_inputs_kernel<unsigned char><<<cdiv(B * HW, 256), 256, 0, s>>>(img_u8, sk_u8, rg_u8, img, region, sk_region, B, HW);
  SE_CUDA_OK(cudaGetLastError());
  return 0;
}
int region_sketch(const float* sketch, const float* region, float* sk_region, int B, int H, int W, cudaStream_t s) {
  const long long HW = (long long)H * W;
  region_inputs_kernel<float><<<cdiv(B * HW, 256), 256, 0, s>>>(nullptr, sketch, region, nullptr, nullptr, sk_region, B, HW);
  SE_CUDA_OK(cudaGetLastError());
  return 0;
}

// test.py:25-27,33-35: (mask*255).astype(uint8); ((x+1)/2*255).astype(uint8) (truncation), CHW->HWC, RGB->BGR
__global__ void to_uint8_kernel(const float* __restrict__ comp, const float* __restrict__ mask, unsigned char* __restrict__ bgr,
                                unsigned char* __restrict__ mk, int B, long long HW) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= B * HW) return;
  const long long b = i / HW, pix = i % HW;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float v = (comp[(b * 3 + c) * HW + pix] + 1.0f) / 2.0f * 255.0f;
    bgr[i * 3 + (2 - c)] = (unsigned char)(int)v;
  }
  if (mk) mk[i] = (unsigned char)(int)(mask[i] * 255.0f);
}

int to_uint8(const float* comp, const float* mask, unsigned char* bgr, unsigned char* mk, int B, int H, int W, cudaStream_t s) {
  const long long HW = (long long)H * W;
  to_uint8_kernel<<<cdiv(B * HW, 256), 256, 0, s>>>(comp, mask, bgr, mk, B, HW);
  SE_CUDA_OK(cudaGetLastError());
  return 0;
}

// debug: number of non-finite bf16 values in a buffer
__global__ void count_nonfinite_kernel(const __nv_bfloat16* __restrict__ x, long long n, unsigned long long* out) {
  long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  unsigned long long c = 0;
  for (; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float v = __bfloat162float(x[i]);
    if (!(fabsf(v) <= 3.0e38f)) ++c;
  }
  if (c) atomicAdd(out, c);
}
long long count_nonfinite_bf16(const void* x, long long n, cudaStream_t s) {
  static unsigned long long* d = nullptr;
  if (!d) cudaMalloc(&d, 8);
  cudaMemsetAsync(d, 0, 8, s);
  count_nonfinite_kernel<<<256, 256, 0, s>>>((const __nv_bfloat16*)x, n, d);
  unsigned long long h = 0;
  cudaMemcpyAsync(&h, d, 8, cudaMemcpyDeviceToHost, s);
  cudaStreamSynchronize(s);
  return (long long)h;
}

// zero-fill helper for padded channel tails
int fill_zero(void* p, size_t bytes, cudaStream_t s) {
  SE_CUDA_OK(cudaMemsetAsync(p, 0, bytes, s));
  return 0;
}

}  // namespace se
