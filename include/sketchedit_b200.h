/*
 * sketchedit_b200 -- C ABI of the B200-native SketchEdit generator forward pass.
 *
 * The reference (zengxianyu/sketchedit) has no FFI / plugin layer: its boundary for this path is the
 * Python nn.Module surface. These entry points are what a binding for that surface calls; each one
 * names the reference interface it replaces. All pointers are plain device pointers (fp32, NCHW,
 * contiguous -- the layout of the torch tensors the reference passes) unless stated otherwise; no
 * torch types cross the boundary. Every function returns 0 on success; on failure it returns non-zero
 * and se_last_error() describes why. `stream` is a cudaStream_t (pass torch's current stream).
 *
 * Kernels are sm_100a only; there is no CPU fallback.
 */
#ifndef SKETCHEDIT_B200_H
#define SKETCHEDIT_B200_H

#ifdef __cplusplus
extern "C" {
#endif

typedef struct se_model se_model;

/* arithmetic / storage mode of a forward call */
enum {
  SE_PREC_BF16_TC = 0,     /* bf16 activations + weights, tcgen05 tensor-core kernels, fp32 accumulation */
  SE_PREC_FP32_EXACT = 1,  /* fp32 activations + weights, CUDA-core fp32 FMA kernels (fp32 parity config) */
  SE_PREC_BF16_DIRECT = 2, /* bf16 activations, CUDA-core kernels (cross-check of the tcgen05 path) */
  SE_PREC_FP32_TC = 3      /* fp32-parity arithmetic ON the tensor cores: activations and weights as fp16 hi + fp16 lo pairs (22
                              significant bits), three tcgen05 products per tap (hi*hi + hi*lo + lo*hi), fp32 accumulation and exact-math
                              epilogue. The fp32 parity config (1e-3) runs here; SE_PREC_FP32_EXACT stays as its cross-check. */
};

/* model options == the reference's command-line flags read on the hot path
 * (reference models/networks/editline_g.py:15-23,28-31 and options/base_options.py:19) */
enum {
  SE_OPT_USE_CAM = 0,        /* --use_cam          (default 1) */
  SE_OPT_POOL_AVG = 1,       /* --pool_type avg    (default 0 = max) */
  SE_OPT_NO_MASK_CC = 2,     /* --no_mask_cc       (default 0) */
  SE_OPT_NO_MASK_COARSE = 3, /* --no_mask_coarse   (default 0) */
  SE_OPT_JOINT_TRAIN_INP = 4 /* --joint_train_inp  (default 1, as in test_celeb.sh / test_places.sh) */
};

const char* se_last_error(void);
int se_abi_version(void);

/* ---- weights: replaces nn.Module parameter ownership + util.load_network
 *      (reference util/util.py:214-225; state_dict keys "<layer>.weight" [cout,cin,k,k], "<layer>.bias" [cout]) */
int se_model_create(se_model** out);
void se_model_destroy(se_model* m);
/* net: 'M' (MDGenerator, reference models/networks/editline2_g.py:14-43) or
 *      'G' (DeepFillC2Generator, reference models/networks/editline_g.py:44-100).
 * weight / bias: HOST fp32 pointers, OIHW. Shapes are validated against the architecture table. */
int se_model_set_layer(se_model* m, char net, const char* layer, const float* weight, const float* bias, int cout, int cin,
                       int ksize);
/* uploads and packs every layer; fails if a layer of either network is missing */
int se_model_finalize(se_model* m);
int se_model_set_option(se_model* m, int option, int value);

/* ---- whole path: replaces EditLine2Model.forward(data, mode='inference')
 *      (reference models/editline2_model.py:107-133 + generate_fake :338-370).
 * image [B,3,H,W] in [-1,1], sketch [B,1,H,W] in {0,1}; H, W multiples of 8 and H/4, W/4 >= 4.
 * Outputs: composed [B,3,H,W], mask [B,1,H,W] (soft). Optional (may be NULL): coarse, fine [B,3,H,W],
 * mask_image [B,3,H,W] (netM image head, only mode='visualize' uses it), mask_bin_out [B,1,H,W].
 * mask_bin_in (optional): use this binarised mask for netG instead of (mask > 0.5). */
int se_forward_inference(se_model* m, const float* image, const float* sketch, int B, int H, int W, int precision,
                         float* composed, float* mask, float* coarse, float* fine, float* mask_image,
                         const float* mask_bin_in, float* mask_bin_out, void* stream);

/* Same forward, outputs written as ONE packed tensor [B,4,H,W] (channels 0-2 composed, channel 3 the soft mask): the
 * layout of the data-parallel output all-gather (SURVEY.md 8e: `[B/n,4,H,W]` shards), so a rank's heads write straight
 * into its slice of the gather buffer and no pack/concat pass exists. */
int se_forward_inference_packed(se_model* m, const float* image, const float* sketch, int B, int H, int W, int precision,
                                float* packed, void* stream);

/* Same forward with the host-side codecs of the reference's test flow moved onto the device: inputs as the dataset reads them
 * before ToTensor/Normalize (reference data/testimage_dataset.py:89-103: image_u8 [B,H,W,3] RGB, sketch_u8 [B,H,W] already resized
 * to the image; on device: x/255 -> (x-0.5)/0.5, sketch > 0), outputs as test.py writes them (reference test.py:25-35:
 * ((x+1)/2*255) and (mask*255) truncated to uint8, HWC, RGB->BGR): bgr_u8 [B,H,W,3], mask_u8 [B,H,W]. 4x fewer bytes each way. */
int se_forward_inference_u8(se_model* m, const unsigned char* image_u8, const unsigned char* sketch_u8, int B, int H, int W,
                            int precision, unsigned char* bgr_u8, unsigned char* mask_u8, void* stream);

/* ---- region inpaint: the user chooses WHERE the edit happens; netM does not run. At inference the reference never takes this
 *      branch of generate_fake (models/editline2_model.py:340-352 external-mask case, :362-368), which its checkpoints were trained
 *      for under --joint_train_inp: mask_inpaint = R, line_inpaint = line_full * R, rm2 = R, netG(x, x, R, R, s*R), then
 *      composed = fine*R + x*(1-R) (:114, :324).
 * image [B,3,H,W] in [-1,1], sketch [B,1,H,W], region R [B,1,H,W] (1 = edit here), both used as given. Outputs: composed
 * [B,3,H,W] (equal to image wherever R = 0); optional (may be NULL) coarse, fine [B,3,H,W]. Model options apply as in
 * se_forward_inference. */
int se_forward_inpaint(se_model* m, const float* image, const float* sketch, const float* region, int B, int H, int W, int precision,
                       float* composed, float* coarse, float* fine, void* stream);

/* Same forward with the codecs of se_forward_inference_u8: image_u8 [B,H,W,3] RGB, sketch_u8 and region_u8 [B,H,W] decoded as
 * s = sketch_u8 > 0, R = region_u8 > 0; output bgr_u8 [B,H,W,3] ((x+1)/2*255 truncated, HWC, RGB->BGR). */
int se_forward_inpaint_u8(se_model* m, const unsigned char* image_u8, const unsigned char* sketch_u8, const unsigned char* region_u8,
                          int B, int H, int W, int precision, unsigned char* bgr_u8, void* stream);

/* ---- netM: replaces MDGenerator.forward(x, guide) -> (mask1, x_stage1)  (editline2_g.py:59-94) */
int se_netM_forward(se_model* m, const float* x, const float* guide, int B, int H, int W, int precision, float* mask1,
                    float* x_stage1 /* may be NULL */, void* stream);

/* ---- netG: replaces DeepFillC2Generator.forward(x, x2, mask, mask2, guide) -> (x_stage1, x_stage2)
 *      (editline_g.py:119-221). mask / mask2 [B,1,H,W]. guide may be NULL = the reference's guide=None (an all-ones
 *      sketch channel, editline_g.py:127-130). */
int se_netG_forward(se_model* m, const float* x, const float* x2, const float* mask, const float* mask2, const float* guide,
                    int B, int H, int W, int precision, float* x_stage1, float* x_stage2, void* stream);

/* ---- operators: replace gen_conv.forward / gen_deconv.forward (reference models/networks/utils.py:25-33, 48-51)
 * for the named layer of the named net. x [B,cin,H,W] -> y [B,cout_after_gate,Ho,Wo]. */
int se_gated_conv_forward(se_model* m, char net, const char* layer, const float* x, int B, int H, int W, int precision,
                          float* y, void* stream);

/* ---- replaces ReduceContextAttentionP1.forward + ReduceContextAttentionP2.forward as netG calls them
 *      (reference models/networks/splitcam.py:57-108,147-174; editline_g.py:203-207):
 * feat [B,C,h,w] (query = key = value source), mask_s [B,1,h,w] hole fraction; out [B,C,h,w].
 * attn (optional, may be NULL) receives the softmax weights [B, L, hs*ws] like cam_1's return value. */
int se_contextual_attention_forward(const float* feat, const float* mask_s, int B, int C, int h, int w, int precision,
                                    float* out, float* attn, void* stream);

/* ---- test.py:25-27 output conversion on device: uint8 HWC BGR image + uint8 mask (truncating) */
int se_outputs_to_uint8(const float* composed, const float* mask, int B, int H, int W, unsigned char* bgr_hwc,
                        unsigned char* mask_u8, void* stream);

/* ---- Pillow's Image.resize((w, h)) with its default filter (BICUBIC) on uint8 HWC images, bit for bit: the resizes of the
 *      reference's demo.py:45,49,68 (to a multiple of 8 and back) on the device. Uses no model.
 * A ragged batch of B images with C = 1 or 3 channels: image i is src_hw[2i] x src_hw[2i+1] (height, width) at byte offset
 * src_off[i] from src and becomes dst_hw[2i] x dst_hw[2i+1] at byte offset dst_off[i] from dst. src_off, src_hw, dst_off and
 * dst_hw are HOST arrays; src and dst are device pointers (the images must not overlap their outputs). One launch per pass
 * (horizontal, then vertical) covers the batch. flags: SE_RESIZE_REVERSE_CHANNELS writes the channels reversed (BGR <-> RGB),
 * images of unchanged size included (those are copied, as Pillow does). The coefficient tables of every (in, out) pair are
 * built on the host the first time the pair is seen on a device and stay cached there. */
enum { SE_RESIZE_REVERSE_CHANNELS = 1 };
int se_resize_u8(const unsigned char* src, const long long* src_off, const int* src_hw, int B, int C, unsigned char* dst,
                 const long long* dst_off, const int* dst_hw, int flags, void* stream);
/* Host only (no device needed): the coefficient tables of one in -> out pass of se_resize_u8. Returns ksize, the weights per
 * output index, or -1 on error. bounds [out][2] = (first source index, tap count); weights [out][ksize] int32 in 22-bit fixed
 * point, zero past the tap count. They are written only if bounds and weights are non-NULL and cap >= out * ksize. */
int se_resize_coeffs(int in, int out, int* bounds, int* weights, int cap);

/* ---- introspection for bench.py */
/* number of kernels this library launched during the most recent forward-type call on this thread */
int se_last_launch_count(void);
/* bytes of device workspace currently held by the model's arena */
long long se_workspace_bytes(se_model* m);
/* when set (default 0), every kernel launch of the forward calls is bracketed by CUDA events on its stream and
 * accounted to a kernel class (kernel + layer shape) with its algorithmic FLOPs / bytes. se_timing_report writes a
 * JSON table of the classes seen since the last se_timing_enable(1) into buf (returns the length needed, -1 on error).
 * Throughput must be measured with timing OFF; bench.py runs one separate instrumented pass for its roofline table. */
int se_timing_enable(int on);
int se_timing_report(char* buf, int cap);

#ifdef __cplusplus
}
#endif
#endif
