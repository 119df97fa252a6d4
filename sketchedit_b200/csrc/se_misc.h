// Glue kernels (se_misc.cu). dt = activation storage type (DT_BF16 / DT_F32).
#pragma once
#include "se_common.cuh"

namespace se {

enum { PACK_IMG_ONE = 0, PACK_IMG_ONE_MINUS_M = 1, PACK_IMG_M = 2 };
enum { HEAD_MASK = 0, HEAD_TANH = 1, HEAD_COARSE = 2, HEAD_FINE = 3 };
enum { RED_MAX = 0, RED_AVG = 1, RED_RNORM = 2 };

int pack8(const float* img, const float* sketch, const float* mask, void* out, int dt, int B, int H, int W, int Wp, int padl,
          int img_mode, float sketch_scale, int write_mask, cudaStream_t s, int img2_mode = -1);   // img2_mode >= 0: channels 5..7 = img * f(mask)
int head(const void* x, int dt, int in_c8, const float* w, const float* bias, int cout, int B, int H, int W, int mode, const float* img,
         const float* mask_bin, const float* mask_soft, float* out_nchw, float* out2, void* out_pack8, int no_mask_coarse,
         int Wp, int padl, long long out_bstride, long long msoft_bstride, unsigned char* out_u8,
         cudaStream_t s);   // strides: elements between images, 0 = dense; out_u8: HEAD_MASK -> mask bytes [B,H,W], HEAD_FINE -> BGR HWC bytes
int head_c8(const void* x, const float* w_host, const float* b_host, int cout, int B, int H, int W, int mode, const float* img,
            const float* mask_bin, const float* mask_soft, float* out_nchw, float* out2, void* out_pack8, int no_mask_coarse, int Wp, int padl,
            long long out_bstride, long long msoft_bstride, unsigned char* out_u8, cudaStream_t s);
int plane_reduce(const void* x, int dt, int B, int HW, int C, int ldx, int c8, int mode, float* out, cudaStream_t s);
int broadcast_channels(const float* v, void* y, int dt, int B, int HW, int C, int ldo, int choff, int c8, cudaStream_t s);
int avgpool4(const float* m, float* out, int B, int H, int W, cudaStream_t s);
int cam_colmask(const float* mask_s, float* out, int B, int h, int w, int hs, int ws, float th, cudaStream_t s);
int cam_pack_k(const void* f, int dt, const float* rnorm, void* out, int B, int h, int w, int C, int ws, int L, int Lpad, cudaStream_t s);
int cam_pack_v(const void* f, int dt, void* out, int B, int h, int w, int C, int ws, int L, int Lpad, cudaStream_t s);
int softmax_rows(const float* S, int lds, void* P, int dt, int ldp, long long rows, int L, cudaStream_t s);
int nchw_to_stem8(const float* x, void* y, int dt, int B, int cin, int H, int W, int Wp, int padl, cudaStream_t s);
int nchw_to_c8_s2d(const float* x, void* y, int B, int C, int H, int W, cudaStream_t s);
int nchw_to_c8(const float* x, void* y, int B, int C, int HW, cudaStream_t s);
int c8_to_nchw(const void* x, float* y, int B, int C, int HW, cudaStream_t s);
int nchw_to_nhwc(const float* x, void* y, int dt, int B, int C, int HW, int ldo, int choff, cudaStream_t s);
int nhwc_to_nchw(const void* x, int dt, float* y, int B, int C, int HW, int ldx, int choff, cudaStream_t s);
int u8_to_inputs(const unsigned char* img_u8, const unsigned char* sk_u8, float* img, float* sk, int B, int H, int W, cudaStream_t s);
// region inpaint inputs (one kernel): uint8 entry -> image, R = region > 0 and s*R planes; float entry -> the s*R plane only
int region_inputs_u8(const unsigned char* img_u8, const unsigned char* sk_u8, const unsigned char* rg_u8, float* img, float* region, float* sk_region,
                     int B, int H, int W, cudaStream_t s);
int region_sketch(const float* sketch, const float* region, float* sk_region, int B, int H, int W, cudaStream_t s);
int to_uint8(const float* comp, const float* mask, unsigned char* bgr, unsigned char* mk, int B, int H, int W, cudaStream_t s);
// split-half twins (se_split.cu): activations stored as fp16 hi + fp16 lo (DT_F16X2)
int pack8_split(const float* img, const float* sketch, const float* mask, void* out, int B, int H, int W, int Wp, int padl, int img_mode,
                float sketch_scale, int write_mask, cudaStream_t s);
int head_split(const void* x, const float* w, const float* bias, int cout, int B, int H, int W, int mode, const float* img, const float* mask_bin,
               const float* mask_soft, float* out_nchw, float* out2, void* out_pack8, int no_mask_coarse, int Wp, int padl, long long obs, long long msbs,
               unsigned char* out_u8, cudaStream_t s);
int plane_reduce_split(const void* x, int B, int HW, int C, int ld, int mode, float* out, cudaStream_t s);
int broadcast_split(const float* v, void* y, int B, int HW, int C, int ld, int choff, cudaStream_t s);
int nchw_to_split(const float* x, void* y, int B, int C, int H, int W, int layout, int Wp, int padl, cudaStream_t s);
int split_to_f32(const void* x, float* y, int B, int C, int HW, int ld, int choff, int nhwc, cudaStream_t s);
int nhwc_f32_to_split(const float* x, void* y, int B, int C, int HW, int ld, int choff, cudaStream_t s);
long long count_nonfinite_bf16(const void* x, long long n, cudaStream_t s);
int fill_zero(void* p, size_t bytes, cudaStream_t s);

}  // namespace se
