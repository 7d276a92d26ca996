/* hitsir_b200 -- C ABI of the B200-native HiT-SIR-pro forward pass.
 *
 * Drop-in boundary for ONE path of CoderLinxin/Single-Image-Super-Resolution-Application:
 * `HiT_SIR.forward` (reference: models/hit_sir_pro.py:1304-1344, constructed at
 * models/hit_sir_pro.py:1091-1265).  The reference has no FFI of its own (it is pure PyTorch);
 * every entry point below therefore names the reference *Python* interface it stands in for, and
 * INTEGRATION.md shows the ctypes binding a maintainer adds (it is what
 * `hitsir_b200.HiT_SIR` uses).
 *
 * Conventions: plain pointers and sizes only (no torch types); every function returns 0 on
 * success and a non-zero status otherwise, with a human-readable message available from
 * hitsir_last_error() (thread-local).  The library never synchronises the device, never
 * changes the current device and launches everything on the caller's stream.  It owns only the
 * packed weights tied to a handle; inputs, outputs and the workspace belong to the caller.
 * There is no CPU path: without an sm_100 device every compute entry point fails.
 */
#ifndef HITSIR_B200_H_
#define HITSIR_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define HITSIR_API __attribute__((visibility("default")))
#else
#define HITSIR_API
#endif

#define HITSIR_MAX_LAYERS 16
#define HITSIR_MAX_DEPTH 16

/* status codes */
enum {
  HITSIR_OK = 0,
  HITSIR_ERR_CUDA = 1,           /* a CUDA call failed (message has the details)                     */
  HITSIR_ERR_INVALID = 2,        /* bad argument / unknown parameter name / wrong element count        */
  HITSIR_ERR_UNSUPPORTED = 3,    /* legal reference configuration this build does not implement        */
  HITSIR_ERR_INPUT_TOO_SMALL = 4,/* reflect padding needs pad < dim (RuntimeError at hit_sir_pro.py:672) */
  HITSIR_ERR_WEIGHTS = 5,        /* forward before all parameters were provided / finalized            */
  HITSIR_ERR_WORKSPACE = 6       /* workspace too small or misaligned                                  */
};

/* upsampler selector: reference constructor argument `upsampler` (hit_sir_pro.py:1116, 1235-1262) */
enum {
  HITSIR_UP_NONE = 0,                /* upsampler=None / '' : x + conv_last(res)   (:1335-1340) */
  HITSIR_UP_PIXELSHUFFLE = 1,        /* 'pixelshuffle'                            (:1313-1319) */
  HITSIR_UP_PIXELSHUFFLEDIRECT = 2,  /* 'pixelshuffledirect'                      (:1320-1325) */
  HITSIR_UP_NEAREST_CONV = 3         /* 'nearest+conv' (x4 only, assert at :1248) (:1326-1334) */
};

/* Mirrors the constructor arguments of HiT_SIR.__init__ (hit_sir_pro.py:1091-1120) that change
 * the forward pass.  Arguments with no effect at inference (img_size, patch_size, drop rates at
 * eval, use_checkpoint, norm_layer=LayerNorm) are handled by the Python mirror. */
typedef struct HitsirConfig {
  int32_t is_mult_size_conv_feat_extract; /* "mulsizeconvextract" */
  int32_t is_channel_spatial_attn;        /* "casa"               */
  int32_t is_fusion;
  int32_t in_chans;                       /* 3 (RGB mean subtracted, :1126-1131) or 1 */
  int32_t embed_dim;                      /* 180 in this build */
  int32_t num_layers;                     /* len(depths) */
  int32_t depths[HITSIR_MAX_LAYERS];
  int32_t num_heads[HITSIR_MAX_LAYERS];   /* 6 in this build */
  int32_t base_win_size[2];               /* square, <= 8 */
  float mlp_ratio;                        /* 2.0 in this build */
  int32_t upscale;
  float img_range;
  int32_t upsampler;                      /* HITSIR_UP_* */
  int32_t num_ratios;
  float hier_win_ratios[HITSIR_MAX_DEPTH];
  int32_t resi_3conv;                     /* resi_connection: 0 = '1conv', 1 = '3conv' (:913-918, :1224-1231) */
  int32_t ape_tokens;                     /* ape=True: (img_size / patch_size)^2 rows of absolute_pos_embed (:1187-1189); 0 = off */
} HitsirConfig;

typedef struct HitsirHandle HitsirHandle;

/* HiT_SIR.__init__ (hit_sir_pro.py:1091).  Binds the handle to the CURRENT CUDA device. */
HITSIR_API int hitsir_create(const HitsirConfig* cfg, HitsirHandle** out);
HITSIR_API void hitsir_destroy(HitsirHandle* h);

/* Names/sizes of the parameters the handle expects == the reference state_dict keys
 * (nn.Module.state_dict(), used by experiment.py:223,260).  hitsir_param_name returns NULL past the end. */
HITSIR_API int hitsir_num_params(const HitsirHandle* h);
HITSIR_API const char* hitsir_param_name(const HitsirHandle* h, int index);
HITSIR_API int64_t hitsir_param_numel(const HitsirHandle* h, int index);

/* nn.Module.load_state_dict(): provide one fp32 tensor by its state_dict key.  `data` may be a
 * device or a host pointer (copied with cudaMemcpyDefault on `stream`); contiguous, `numel` floats. */
HITSIR_API int hitsir_set_param(HitsirHandle* h, const char* name, const float* data, int64_t numel, void* stream);
/* Pack weights (bf16 K-major operands, padded) and precompute the pooled relative-position bias
 * tables (hit_sir_pro.py:477-503 hoisted out of the forward).  Call after all parameters are set
 * and again whenever any of them changed. */
HITSIR_API int hitsir_finalize_weights(HitsirHandle* h, void* stream);

/* Scratch memory needed by hitsir_forward for a (B,H,W) input; 256-byte aligned base required. */
HITSIR_API int hitsir_workspace_bytes(const HitsirHandle* h, int B, int H, int W, size_t* bytes);

/* HiT_SIR.forward (hit_sir_pro.py:1304-1344): x (B,in_chans,H,W) fp32 NCHW on the device ->
 * y (B,in_chans,H*upscale,W*upscale) fp32 NCHW on the device.  Asynchronous on `stream`. */
HITSIR_API int hitsir_forward(HitsirHandle* h, const float* x, float* y, int B, int H, int W,
                   void* workspace, size_t workspace_bytes, void* stream);

/* ---- exact multi-GPU sharding of ONE frame by rows (SURVEY.md 8f-1) --------------------------------------------------------------
 * The reference always runs whole frames (test_experiment.py:75, experiments/experiment.py:743) and its casa pools (hit_sir_pro.py:348-349)
 * and UnionAttention row / column statistics (:124-130) span the frame, so halo TILES are not the full-frame forward.  In band mode every
 * GPU computes the rows [row0, row0 + H) of the frame -- band boundaries are multiples of 192 = lcm of the window sizes, so no window
 * straddles two bands -- and the library asks the caller for exactly two kinds of exchange while it enqueues the forward:
 *   halo:       the `halo_rows` rows above / below the `rows` core rows of a row-major buffer at workspace offset `ws_offset` must be
 *               filled with the neighbour band's adjacent core rows (1 row for the 3x3 convolutions and the casa / UnionAttention
 *               statistic maps, 2 rows of the FFN hidden map for the depthwise 5x5).  Every band lays its workspace out identically
 *               (layout_h = the largest band height), so the neighbour's buffer is at the same offset of ITS workspace.
 *   allreduce:  element-wise SUM of n_sum floats and MAX of n_max floats over all bands (casa global pools, UnionAttention column
 *               statistics), in place.  Called whenever the pointer is non-NULL, also for a frame that is a single band (the
 *               reduction is then the identity; callers use it to observe the statistics).
 * Both run on the host thread that called hitsir_forward_band and must order their work on `stream`.  B = 1. */
typedef int (*hitsir_halo_fn)(void* ctx, int64_t ws_offset, int64_t row_bytes, int32_t rows, int32_t halo_rows, void* stream);
typedef int (*hitsir_allreduce_fn)(void* ctx, int64_t sum_offset, int64_t n_sum, int64_t max_offset, int64_t n_max, void* stream);
typedef struct HitsirBand {
  int32_t frame_h;       /* rows of the whole frame                                              */
  int32_t row0;          /* first frame row of this band (a multiple of 192)                      */
  int32_t layout_h;      /* largest band height of the frame: common workspace layout             */
  int32_t has_top;       /* a neighbour band exists above / below                                 */
  int32_t has_bottom;
  hitsir_halo_fn halo;
  hitsir_allreduce_fn allreduce;
  void* ctx;
} HitsirBand;
HITSIR_API int hitsir_workspace_bytes_band(const HitsirHandle* h, int layout_h, int W, size_t* bytes);
/* x_frame: the WHOLE LR frame (1, in_chans, frame_h, W) fp32 NCHW on this device (the 9x9 entry footprint reads across the band edge);
 * y_band: (1, in_chans, s*H, s*W) = the band's rows of the output. */
HITSIR_API int hitsir_forward_band(HitsirHandle* h, const float* x_frame, float* y_band, int H, int W, const HitsirBand* band,
                        void* workspace, size_t workspace_bytes, void* stream);

/* Same call with HOST buffers (pinned recommended): copies x host->device, runs the forward,
 * copies y device->host, all on `stream`; `dev_x`/`dev_y` are caller-provided device staging
 * buffers of B*C*H*W and B*C*sH*sW floats.  Returns after enqueueing; the caller synchronises. */
HITSIR_API int hitsir_forward_host(HitsirHandle* h, const float* host_x, float* host_y, int B, int H, int W,
                        float* dev_x, float* dev_y, void* workspace, size_t workspace_bytes, void* stream);

/* The image-file round trip of test_experiment.py:70-77 on the device: `x_hwc` is a PIL-style uint8 image batch [B,H,W,C]
 * (utils/utils.py:143-145 to_tensor: value / 255), the result is clip(0,1) (experiments/experiment.py:746-748) converted like
 * torchvision's to_pil_image (value * 255, truncated) into `y_hwc` [B,sH,sW,C].  `dev_x`/`dev_y` are caller-provided fp32 staging
 * buffers of B*C*H*W and B*C*sH*sW floats; all pointers are device pointers. */
HITSIR_API int hitsir_forward_u8(HitsirHandle* h, const uint8_t* x_hwc, uint8_t* y_hwc, int B, int H, int W,
                      float* dev_x, float* dev_y, void* workspace, size_t workspace_bytes, void* stream);

/* ---- x8 geometric self-ensemble (the "+" test mode of EDSR+ / RCAN+ / SwinIR+, BasicSR's test_selfensemble) ------------------------
 * Transform k = 0..7 in BasicSR's order: bit 0 flips W, bit 1 flips H, bit 2 swaps H and W, applied in that order.  The result is
 *   y = (((((((z0' + z1') + z2') + z3') + z4') + z5') + z6') + z7') * 0.125f,   zk' = T_k^-1(forward(T_k(x)))
 * summed in this fixed ascending order in fp32.  The forward runs `group` transforms of the B images as ONE batch of group*B images
 * (8 / group rounds of: transform kernel, forward, combine kernel).  group is 1, 2, 4 or 8, and 8 (both orientations in one batch)
 * needs H == W; group*B*H*W*16 < 2^31.  Taps and injections are refused (HITSIR_ERR_UNSUPPORTED).
 * hitsir_workspace_bytes_x8: the larger forward workspace of group*B images at H x W and at W x H, plus the transformed inputs, the
 * outputs of one group and the fp32 accumulator of the uint8 entry; one allocation serves both entries. */
HITSIR_API int hitsir_workspace_bytes_x8(const HitsirHandle* h, int B, int H, int W, int group, size_t* bytes);
/* x (B,in_chans,H,W) fp32 NCHW -> y (B,in_chans,sH,sW) fp32 NCHW, both on the device; y is also the accumulator. */
HITSIR_API int hitsir_forward_x8(HitsirHandle* h, const float* x, float* y, int B, int H, int W, int group,
                      void* workspace, size_t workspace_bytes, void* stream);
/* hitsir_forward_u8's image round trip around the self-ensemble: bit-identical to hitsir_f32nchw_to_u8hwc of hitsir_forward_x8's
 * result for x_hwc / 255 in NCHW. */
HITSIR_API int hitsir_forward_x8_u8(HitsirHandle* h, const uint8_t* x_hwc, uint8_t* y_hwc, int B, int H, int W, int group,
                         void* workspace, size_t workspace_bytes, void* stream);

/* The exit conversion alone: clip(0,1) (experiments/experiment.py:746-748) and torchvision's to_pil_image (value * 255, truncated) of
 * an fp32 NCHW batch [B,C,H,W] into uint8 HWC [B,H,W,C], both on the device.  Used before the multi-GPU output gather: a quarter of
 * the fp32 bytes cross NVLink.  Needs no handle; asynchronous on `stream`. */
HITSIR_API int hitsir_f32nchw_to_u8hwc(const float* src, uint8_t* dst, int B, int C, int H, int W, void* stream);
/* The same with BasicSR's tensor2img rounding (basicsr/utils/img_util.py, uint8 output): clip(0,1), value * 255 in fp32, rounded half
 * to even, of an fp32 NCHW batch [B,C,H,W] into uint8 HWC [B,H,W,C].  Needs no handle; asynchronous on `stream`. */
HITSIR_API int hitsir_f32nchw_to_u8hwc_round(const float* src, uint8_t* dst, int B, int C, int H, int W, void* stream);

/* The entry conversion alone, the mirror of hitsir_f32nchw_to_u8hwc: torchvision's to_tensor (utils/utils.py:143-145: value / 255 in
 * fp32) of a uint8 HWC batch [B,H,W,C] into fp32 NCHW [B,C,H,W], both on the device; the conversion hitsir_forward_u8 applies to its
 * input.  Needs no handle; asynchronous on `stream`. */
HITSIR_API int hitsir_u8hwc_to_f32nchw(const uint8_t* src, float* dst, int B, int C, int H, int W, void* stream);

/* ---- bicubic resizing: the LR synthesis of the evaluation (datasets/dataset.py:51-91) and the "Bicubic" baseline ------------------
 * Two standard definitions over one separable resampler (horizontal pass, then vertical) with per-axis tap tables that the call builds
 * on the device in `scratch` (hitsir_resize_scratch_bytes(mode, H, W, outH, outW) bytes of device memory, 4-byte aligned): no host copy, so a call
 * can be captured in a CUDA graph.  No atomics (bitwise reproducible; an image's result does not depend on the rest of the batch),
 * asynchronous on `stream`, no handle.  Null pointers, an empty batch, a zero-sized input or output and C not in {1, 3} are
 * HITSIR_ERR_INVALID, and so is a downscale so strong that a tile's tap tables outgrow a CTA's shared memory (a factor above ~150). */
enum { HITSIR_RESIZE_PIL = 0, HITSIR_RESIZE_MATLAB = 1 };
/* For HITSIR_RESIZE_MATLAB pass outH = ceil(H * scale), outW = ceil(W * scale); an axis that shrinks to one sample is sized for
 * scale >= 1 / max(its length, 16), and a smaller scale is HITSIR_ERR_INVALID.  0 for arguments the entries refuse. */
HITSIR_API int64_t hitsir_resize_scratch_bytes(int mode, int H, int W, int outH, int outW);
/* Pillow 12.2 Image.resize((outW, outH), Image.BICUBIC), modes "L" (C = 1) and "RGB" (C = 3), box and reducing_gap at their defaults:
 * bit-exact.  Cubic a = -0.5 with support 2 * max(in/out, 1), weights normalised in double and rounded to 22-bit fixed point, int32
 * sums, uint8 intermediate (libImaging/Resample.c).  uint8 HWC [B,H,W,C] -> uint8 HWC [B,outH,outW,C]. */
HITSIR_API int hitsir_resize_u8_pil(const uint8_t* src_hwc, uint8_t* dst_hwc, int B, int H, int W, int C, int outH, int outW, void* scratch,
                         void* stream);
/* MATLAB imresize(x, scale, 'bicubic') as BasicSR's calculate_weights_indices + imresize compute it: cubic a = -0.5, antialiased
 * (kernel width 4 / scale) when scale < 1, half-sample symmetric boundary, output ceil(H * scale) x ceil(W * scale).  Weights in fp64
 * rounded to fp32, fp32 FMA accumulation in tap order: within a bound of the fp64 result that tests/resize_ref.py derives, not
 * bit-exact to BasicSR (fp32 weights, unspecified summation order).  fp32 NCHW [B,C,H,W] -> fp32 NCHW, values not clipped. */
HITSIR_API int hitsir_resize_f32_matlab(const float* src_nchw, float* dst_nchw, int B, int C, int H, int W, double scale, void* scratch,
                             void* stream);

/* The evaluation metric around the path on the device (experiments/experiment.py:436-463, called per batch from :743-755): both fp32
 * NCHW batches [B,3,H,W] in [0,1] are converted to the Y channel of YCbCr exactly as utils/utils.py:170-186 does
 * (16/255 + (65.738 R + 129.057 G + 25.064 B) / 256, fp32), `sr` clipped to [0,1] first when clip_sr != 0 (experiment.py:746-748),
 * and mse_out[b] (device, double) receives the mean squared Y difference of image b: PSNR_b = 10 log10(1 / mse_out[b])
 * (skimage.metrics.peak_signal_noise_ratio, data_range=1).  `scratch`: device buffer of hitsir_psnr_y_scratch_doubles(B,H,W) doubles.
 * Fixed-order reduction (bitwise reproducible); asynchronous on `stream`; needs no handle. */
HITSIR_API int64_t hitsir_psnr_y_scratch_doubles(int B, int H, int W);
HITSIR_API int hitsir_psnr_y(const float* sr, const float* hr, int B, int H, int W, int clip_sr, double* scratch, double* mse_out,
                  void* stream);

/* The evaluation's second metric on the device (experiments/experiment.py:575-640): per-image mean SSIM of the Y channels,
 * skimage.metrics.structural_similarity(hr_y, sr_y, data_range=1) of scikit-image 0.24.  Y and the clip of `sr` as hitsir_psnr_y.
 * With x = Y(hr), y = Y(sr) and window means (weighted by the window) ux, uy, uxx, uyy, uxy of x, y, x*x, y*y, x*y:
 *   vx = cn (uxx - ux^2),  vy = cn (uyy - uy^2),  vxy = cn (uxy - ux uy)
 *   S  = ((2 ux uy + C1)(2 vxy + C2)) / ((ux^2 + uy^2 + C1)(vx + vy + C2)),  C1 = 0.01^2, C2 = 0.03^2,
 * and ssim_out[b] (device, double) is the mean of S over the interior [p, H-p) x [p, W-p), p = (win-1)/2, where every window lies
 * inside the image.  Windows: gaussian == 0 -> uniform 7 x 7 (skimage's default); gaussian != 0 -> Gaussian sigma = 1.5 truncated at
 * 3.5 sigma, 11 x 11, taps exp(-x^2 / (2 sigma^2)) normalised, x = -5..5 (gaussian_weights=True).  sample_cov != 0 -> cn = win^2 /
 * (win^2 - 1), for the Gaussian window too, as skimage does (use_sample_covariance=True, its default); 0 -> cn = 1 (Wang et al.).
 * Products are formed in fp32, window sums in double rounded to fp32, S in fp32 as skimage writes it (ssim(x, x) is exactly 1).
 * H or W smaller than the window is HITSIR_ERR_INVALID (skimage raises ValueError).  `scratch`: device buffer of
 * hitsir_ssim_y_scratch_doubles(B,H,W,gaussian) doubles.  Fixed-order reduction (bitwise reproducible, independent of the other images of
 * the batch); asynchronous on `stream`; needs no handle. */
HITSIR_API int64_t hitsir_ssim_y_scratch_doubles(int B, int H, int W, int gaussian);
HITSIR_API int hitsir_ssim_y(const float* sr, const float* hr, int B, int H, int W, int clip_sr, int gaussian, int sample_cov,
                  double* scratch, double* ssim_out, void* stream);

/* The metrics of published SR tables: BasicSR 1.4.2's calculate_psnr and calculate_ssim (basicsr/metrics/psnr_ssim.py, with
 * to_y_channel of basicsr/metrics/metric_util.py and bgr2ycbcr of basicsr/utils/color_util.py) of two uint8 RGB HWC batches
 * [B,H,W,3] on the device (SR rounded to uint8 first, as tensor2img does: hitsir_f32nchw_to_u8hwc_round).
 *   crop:   crop_border pixels are dropped on every side (none when 0).
 *   planes: y_only != 0 -> one plane, BasicSR's Y on the 0-255 scale: t = fp32(v) / 255 (fp32), y = ((24.966 t_B + 128.553 t_G)
 *           + 65.481 t_R) + 16 (double), Y = fp32(fp32(y / 255) * 255); y_only == 0 -> the three colour channels.
 *   mse_out[b] = the mean over every kept value of (sr - hr)^2 in double: PSNR_b = 10 log10(255^2 / mse_out[b]), +inf when 0.  In RGB
 *           mode the squares are integers summed exactly, so mse_out equals numpy's bit for bit.
 *   ssim_out[b] = per plane, the mean over the valid region [5, Hc-5) x [5, Wc-5) of the crop of
 *           S = ((2 mu1 mu2 + c1)(2 s12 + c2)) / ((mu1^2 + mu2^2 + c1)(s11 + s22 + c2)),  c1 = (0.01 * 255)^2, c2 = (0.03 * 255)^2,
 *           with window means under outer(k, k), k = cv2.getGaussianKernel(11, 1.5), and s = E[ab] - mu_a mu_b; then the mean of the
 *           planes in BasicSR's BGR order ((B + G) + R) / 3.  Double throughout; direct (separable) window sums rather than
 *           cv2.filter2D's DFT, so within a derived per-image bound of BasicSR (1e-13 to 1e-11) rather than bit-exact;
 *           ssim(x, x) is exactly 1.
 * Null pointers, B outside 1..65535, crop_border < 0 and H - 2 crop_border < 11 or W - 2 crop_border < 11 (BasicSR returns nan with a
 * warning) are HITSIR_ERR_INVALID.  `scratch`: device buffer of hitsir_basicsr_metrics_scratch_doubles(B,H,W,crop_border,y_only) doubles
 * (0 for arguments the entry refuses).  No host copy (graph-capturable), fixed-order reduction (bitwise reproducible, independent of the
 * other images of the batch); asynchronous on `stream`; needs no handle. */
HITSIR_API int64_t hitsir_basicsr_metrics_scratch_doubles(int B, int H, int W, int crop_border, int y_only);
HITSIR_API int hitsir_psnr_ssim_basicsr(const uint8_t* sr_hwc, const uint8_t* hr_hwc, int B, int H, int W, int crop_border, int y_only,
                             double* scratch, double* mse_out, double* ssim_out, void* stream);

/* Test hook standing in for PyTorch forward hooks on reference sub-modules: the next
 * hitsir_forward copies the named intermediate activation (fp32, NHWC, real channels only) into
 * `dst` (device) and, when `stop` != 0, returns right after producing it.  Names: "shallow",
 * "embed", "block<i>.<j>.qkv", "block<i>.<j>.scc", "block<i>.<j>.attn", "block<i>.<j>.fc1" (GELU(fc1), 360 channels), "block<i>.<j>",
 * "layer<i>", "norm", "conv_after_body", "fused", "conv_before_upsample", "up1", "up2", "hr".
 * Pass name = NULL to clear. */
HITSIR_API int hitsir_set_tap(HitsirHandle* h, const char* name, float* dst, int64_t dst_floats, int stop);

/* Test hook standing in for a PyTorch forward PRE-hook that replaces a sub-module's input (nn.Module.register_forward_pre_hook):
 * the next hitsir_forward calls overwrite the named activation with `src` (device, fp32, NHWC, [B*H*W, 180]) right before it is
 * consumed.  Names: "block<i>.<j>.in" (the token stream entering HierarchicalTransformerBlock i.j, hit_sir_pro.py:676) and
 * "fused" (the input of the reconstruction stage, :1313-1340).  Together with hitsir_set_tap it isolates one stage, which is how the
 * index work (reflect padding :664-674, window partition / reverse :236-271, nearest upsampling :1331-1332, PixelShuffle :1024-1062)
 * is checked bit for bit.  `src` must stay valid until cleared; pass name = NULL to clear. */
HITSIR_API int hitsir_set_inject(HitsirHandle* h, const char* name, const float* src, int64_t src_floats);

/* The pooled relative-position bias of SCC block (layer, block): `relative_position_bias` of hit_sir_pro.py:477-503, fp32
 * [6 heads][L = w*w tokens][Lb = min(w,8)^2 pooled cells], as precomputed by hitsir_finalize_weights (the reference rebuilds it on
 * every forward).  Copies `dst_floats` = 6*L*Lb floats to `dst` (host or device) on `stream`. */
HITSIR_API int hitsir_get_bias_table(HitsirHandle* h, int layer, int block, float* dst, int64_t dst_floats, void* stream);

/* Number of kernels the last hitsir_forward launched (bench.py's gpu_launches); for hitsir_forward_x8* the whole call. */
HITSIR_API int64_t hitsir_last_launch_count(const HitsirHandle* h);

/* Per-category CUDA-event timing of the launches inside hitsir_forward (events on the caller's stream, no
 * synchronisation added).  Enable, run forwards, synchronise the stream yourself, then read the totals
 * accumulated since the last hitsir_profile_enable call.  Used by bench.py for the live roofline numbers. */
HITSIR_API int hitsir_profile_enable(HitsirHandle* h, int on);
HITSIR_API int hitsir_profile_num_categories(const HitsirHandle* h);
HITSIR_API int hitsir_profile_get(HitsirHandle* h, int index, const char** name, double* total_ms, int64_t* launches);

/* "umma" (tcgen05 path with TMA-staged epilogues) is the only backend.  Any other name returns HITSIR_ERR_INVALID, and
 * hitsir_last_error() names the rejected backend. */
HITSIR_API int hitsir_set_gemm_backend(HitsirHandle* h, const char* backend);

HITSIR_API const char* hitsir_last_error(void);
HITSIR_API const char* hitsir_version(void);

#ifdef __cplusplus
}
#endif
#endif /* HITSIR_B200_H_ */
