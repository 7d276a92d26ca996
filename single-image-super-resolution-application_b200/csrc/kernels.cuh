// Launch prototypes of the non-GEMM kernels (glue.cu, scc.cu, pack.cu).
#pragma once
#include "gemm.cuh"

namespace hitsir {

constexpr int kC = 180;        // embedding width of HiT-SIR-pro
constexpr int kCp = 192;       // padded to a multiple of 64 for TMA / UMMA K blocks
constexpr int kHalf = 90;      // q | v split (hit_sir_pro.py:569-570)
constexpr int kHeads = 6;
constexpr int kHd = 15;        // head dim = C / (2*heads)
constexpr int kHid = 360;      // ConvFFN hidden width (mlp_ratio 2)
constexpr int kHidp = 384;

// ---- glue.cu ---------------------------------------------------------------------------
// NCHW fp32 image -> im2col rows [N, Kp] bf16 of ((x - mean) * img_range), footprint f x f, zero padded
// band mode: rows [y0, y0 + H) of a frame with Hf rows are converted (x is the whole frame); y0 = 0, Hf = 0 -> the whole image
int launch_entry_im2col(const float* x, bf16* a0, int B, int H, int W, int in_ch, int f, int Kp,
                        const float* mean3, float img_range, cudaStream_t st, int y0 = 0, int Hf = 0);
// LayerNorm over rows of fp32 [N,180] -> bf16 [N,192] (pad zero) and/or fp32 [N,180]
// add (optional): fp32 [add_rows, 180] added after the normalisation, row index modulo add_rows (absolute position embedding)
int launch_ln_rows(const float* x, const float* gamma, const float* beta, bf16* out_bf16, float* out_f32, long long N, cudaStream_t st,
                   const float* add = nullptr, long long add_rows = 0);
// ffn_tail.cu: dwconv5 + GELU + input fused with fc2 + LayerNorm + residual (x updated in place); tm_w2 = packed fc2 weights, box {64, 192}
// Optional by-product of ffn_tail: the casa statistics of the block output for the NEXT block (padded to Hp x Wp there):
// cavg/cmax [B*H*W], part_sum/part_max [B * tiles][180] with tiles = ceil(H/8) * ceil(W/16) 8x16-pixel tiles per image
struct FfnStats { float* cavg; float* cmax; float* part_sum; float* part_max; int Hp, Wp; };
inline int ffn_tiles_per_image(int H, int W) { return cdiv(H, kConvTileH) * cdiv(W, kConvTileW); }
// dw_tbl_mma (launch_pack_dw_mma from the fp32 [26][384] tap-major table): the depthwise taps as B-fragment words of the tensor-core
// conv, [384 channels][28 words]: bf16(w) in the low (c even) / high (c odd) half in MMA pairing order, word 26 = fp32 bias bits (pack.cu)
int launch_pack_dw_mma(const float* dw_tbl, uint32_t* out, cudaStream_t st);
// shadow (only without stats): bf16 copy [B*H*W][192] of the updated stream, written by the kernel's statistics warp
// w2_img (launch_pack_w2_image): the packed fc2 weights [192][384] re-laid as six contiguous SWIZZLE_128B operand images [192 rows x 64 k]
// (24 KB each), so that a slice is one bulk copy instead of 192 TMA rows
int launch_pack_w2_image(const bf16* w2_packed, uint8_t* img, cudaStream_t st);
// band (optional, exact row sharding of one frame): h1 has `halo` valid rows above/below, statistics use frame row yg0 + y of Hf rows
struct FfnBand { int halo, yg0, Hf; };
int launch_ffn_tail(const bf16* h1, const uint32_t* dw_tbl_mma, const uint8_t* w2_img, const float* b2, const float* gamma,
                    const float* beta, float* x, int B, int H, int W, const FfnStats* stats, bf16* shadow, int num_sms, cudaStream_t st,
                    const FfnBand* band = nullptr);
// uint8 HWC <-> fp32 NCHW entry / exit (to_tensor: /255; clip(0,1) then to_pil_image: *255 truncated)
int launch_u8hwc_to_f32nchw(const uint8_t* in, float* out, int B, int H, int W, int C, cudaStream_t st);
int launch_f32nchw_to_u8hwc(const float* in, uint8_t* out, int B, int H, int W, int C, cudaStream_t st);
// the same with BasicSR's tensor2img rounding: clip(0,1), fp32 * 255, round half to even
int launch_f32nchw_to_u8hwc_round(const float* in, uint8_t* out, int B, int H, int W, int C, cudaStream_t st);
// perm != 0: column c is read from the head-padded position scc_pos(c)
int launch_f32_to_f32_tap(const void* src, int src_is_bf16, int ld_src, float* dst, long long rows, int cols, int perm, cudaStream_t st);
// out_bf16[N,192] = bf16(a) (pad 0): GEMM operand shadow of the fp32 stream
int launch_cast_rows_bf16(const float* a, bf16* out, long long N, cudaStream_t st);
// out_bf16[N,192] = bf16(a + b) (fusion disabled path, hit_sir_pro.py:1153)
int launch_add_to_bf16(const float* a, const float* b, bf16* out, long long N, cudaStream_t st);

// ---- ensemble.cu (x8 geometric self-ensemble; transform k: bit 0 flips W, bit 1 flips H, bit 2 swaps H and W, in that order) ----
// x fp32 NCHW [B,C,H,W] (or x_u8hwc uint8 [B,H,W,C], /255 as launch_u8hwc_to_f32nchw; the other pointer is nullptr) -> xt [g*B,C,H',W']
// with image kk*B + b = T_{k0+kk}(image b); [k0, k0+g) stays on one side of k = 4 unless H == W
int launch_x8_entry(const float* x, const uint8_t* x_u8hwc, float* xt, int B, int C, int H, int W, int k0, int g, cudaStream_t st);
// acc [B,C,Hd,Wd] (+)= T_k^-1(z_k) for k = k0 .. k0+g-1 in ascending order, z [g*B,C,..] transform-major; first: acc starts from the
// first term; last: * 0.125f, and y_u8hwc != nullptr writes uint8 [B,Hd,Wd,C] as launch_f32nchw_to_u8hwc instead of acc
int launch_x8_combine(const float* z, float* acc, uint8_t* y_u8hwc, int B, int C, int Hd, int Wd, int k0, int g, int first, int last, cudaStream_t st);

// ---- metrics.cu (evaluation metrics of two batches, per image) ----
// per-image mean squared difference of the YCbCr Y channels of two [0,1] fp32 NCHW RGB batches (utils/utils.py:170-186, experiment.py:436-463)
long long psnr_y_chunks(int H, int W);
int launch_psnr_y(const float* sr, const float* hr, int B, int H, int W, int clip, double* partial, double* mse, cudaStream_t st);
// Y-channel SSIM of two [0,1] fp32 NCHW RGB batches, skimage structural_similarity(hr_y, sr_y, data_range=1)
// window radius 3 (uniform 7x7) or 5 (Gaussian sigma 1.5, 11 taps); tiles per image of the interior, 0 when H or W < the window
int ssim_y_radius(int gaussian);
long long ssim_y_tiles(int H, int W, int gaussian);
// partial: B * ssim_y_tiles doubles; ssim[b] = mean of the SSIM map over the interior of image b
int launch_ssim_y(const float* sr, const float* hr, int B, int H, int W, int clip, int gaussian, int sample_cov, double* partial, double* ssim,
                  cudaStream_t st);
// BasicSR 1.4.2's calculate_psnr / calculate_ssim of two uint8 RGB HWC batches (crop_border, test_y_channel = y_only).
// basicsr_metrics_check: 0 when B, the shape and the crop are supported, else 1 with the error message set.
int basicsr_metrics_check(int B, int H, int W, int crop);
long long basicsr_metrics_scratch_doubles(int B, int H, int W, int crop, int y_only);
int launch_psnr_ssim_basicsr(const uint8_t* sr, const uint8_t* hr, int B, int H, int W, int crop, int y_only, double* scratch, double* mse,
                             double* ssim, cudaStream_t st);

// ---- resize.cu (bicubic resizing: Pillow's Image.resize(BICUBIC) on uint8 HWC, MATLAB imresize as BasicSR computes it on fp32 NCHW) ----
// 0 when the shapes (and scale, matlab) are within what the kernel supports, else 1 with the error message set
int resize_check(int matlab, int C, int H, int W, int outH, int outW, double scale);
long long resize_scratch_bytes(int matlab, int H, int W, int outH, int outW);
int launch_resize_pil(const uint8_t* src, uint8_t* dst, int B, int H, int W, int C, int outH, int outW, void* scratch, cudaStream_t st);
int launch_resize_matlab(const float* src, float* dst, int B, int C, int H, int W, double scale, int outH, int outW, void* scratch,
                         cudaStream_t st);

// ---- casa (SpatialChannelAttention, hit_sir_pro.py:338-359) ------------------------------
struct CasaW {
  const float* w1; const float* b1;      // linear1: Conv2d(1,C,3) as [9][C], [C]
  const float* w2; const float* b2;      // linear2
  const float* l1f_w; const float* l1f_b;   // [18][180], [18]
  const float* l1s_w; const float* l1s_b;   // [180][18], [180]
  const float* l2f_w; const float* l2f_b;
  const float* l2s_w; const float* l2s_b;
  const uint32_t* bfrag;                 // linear1/linear2 as split-bf16 MMA B fragments (launch_pack_casa_bfrag); required when casa is on
};
int casa_bfrag_words();
int launch_pack_casa_bfrag(CasaW w, uint32_t* img, cudaStream_t st);
struct PadGeom {
  int B, H, W, Hp, Wp;     // real and reflect-padded sizes
  // band mode (one frame sharded by rows, zero-initialised = off): this band starts at frame row y0 of a frame with Hf rows padded to
  // Hpf; `top` / `bot` say that the per-pixel statistic maps carry one valid halo row of the neighbour band above / below
  int y0, Hf, Hpf, top, bot;
};
// F.pad 'reflect' (hit_sir_pro.py:672): source index of padded index i in [0, 2n - 1)
__device__ __forceinline__ int reflect_src(int i, int n) { return i < n ? i : 2 * (n - 1) - i; }
// number of positions of the padded axis [0, np) that read source index i: padded ip in [n, np) mirrors to 2(n-1) - ip.  The casa pool
// statistics of sca_stats (glue.cu) and of the ffn_tail by-product both weight pixels by it, so both kernels give the same pools.
__device__ __forceinline__ int reflect_mult(int i, int n, int np) { return 1 + ((i >= 2 * (n - 1) - (np - 1) && i <= n - 2) ? 1 : 0); }
// per padded pixel channel mean / max + deterministic per-image per-channel (sum, max) partials
int launch_sca_stats(const float* x, PadGeom g, float* cavg, float* cmax, float* part_sum, float* part_max, int nparts, cudaStream_t st);
int launch_sca_mlp(const float* part_sum, const float* part_max, int nparts, PadGeom g, CasaW w, float* s1, float* s2, cudaStream_t st);
// t[b,yp,xp,:] = x[reflect src] (+ casa gate)  -> bf16 [B*Hp*Wp, 192]
int launch_qkv_build(const float* x, PadGeom g, int casa, const float* cavg, const float* cmax, const float* s1, const float* s2,
                     CasaW w, bf16* t, cudaStream_t st);

// ---- scc_umma.cu (SCC.forward without proj, hit_sir_pro.py:542-596) ---------------------------
// Head-padded token layout of the window tokens T and of the SCC output: reference channel
// c = half*90 + head*15 + j (half 0 = q / out_s, half 1 = v / out_c, :569-570, :596) sits at position
// half*96 + head*16 + j.  The q pads of T (positions 16h+15) hold the constant 1 (k-gen bias rider), the v pads are 0.
__host__ __device__ inline int scc_pos(int c) { const int half = c / kHalf, r = c - half * kHalf; return half * 96 + (r / kHd) * 16 + r % kHd; }
__host__ __device__ inline int scc_chan(int p) { const int half = p / 96, r = p - half * 96; return (r & 15) == 15 ? -1 : half * kHalf + (r >> 4) * kHd + (r & 15); }
// Token tiles of a window: bx x by pixels = TT tokens (TMA box), row-major tiles_x x (tiles/tiles_x) per window
struct SccTile { int bx, by, TT, tiles_x, tiles; };
__host__ __device__ inline SccTile scc_tile(int w) {
  if (w == 4) return SccTile{4, 4, 16, 1, 1};
  if (w == 8) return SccTile{8, 8, 64, 1, 1};
  if (w >= 16 && w <= 64 && w % 16 == 0) return SccTile{16, 8, 128, w / 16, (w / 16) * (w / 8)};
  return SccTile{0, 0, 0, 0, 0};
}
struct SccW {
  const float* wk1; const float* bk1;    // k_generate1 [15][15], [15]
  const float* wk2; const float* bk2;    // k_generate2
  const float* wsl; float* bsl_dev;      // spatial_linear weight [r*r]; bias read from device (1 float)
  const float* bias_tbl;                 // pooled relative-position bias [6][L][Lb]
  const uint8_t* pool_img;               // weights-only UMMA operand images (scc_umma.cu); pool_img: r > 1 only
  const uint8_t* bias_img;
  const uint8_t* w_img;
};
struct SccGeom {
  PadGeom pg;
  int w, base, r;      // window, pooled grid side (min(w,8)), w/base
  int L, Lb;
  int nWy, nWx;        // windows per image
};
size_t scc_pool_image_bytes(int w);
size_t scc_bias_image_bytes(int w);
// pool_img == nullptr skips the pool image (r = 1: scc_dense reads only the bias and k-gen images)
int launch_scc_images(const SccW& w, int win, int base, uint8_t* pool_img, uint8_t* bias_img, uint8_t* w_img, cudaStream_t st);
// windows with pooling ratio r > 1 (scc_dense serves r = 1)
int launch_scc_umma(const bf16* t, const SccGeom& g, const SccW& w, bf16* out, int num_sms, cudaStream_t st);
// scc_dense.cu: windows of 4x4 / 8x8 tokens (pooling ratio 1), several windows per 128-token tile
int launch_scc_dense(const bf16* t, const SccGeom& g, const SccW& w, bf16* out, int num_sms, cudaStream_t st);

// ---- fusion (UnionAttention / Fusion, hit_sir_pro.py:104-162) -------------------------------------
struct UaW {
  const float* c1_w; const float* c1_b;   // conv1 [1][2][3][3], [1]
  const float* c2_w; const float* c2_b;
  const float* c3_w; const float* c3_b;
};
// stats of X = a (+ b if b != nullptr) over channels / rows / columns
// Hf (band mode) = rows of the whole frame: havg holds sum / Hf of the band's rows, so that an all-reduce SUM over the bands is the mean
int launch_ua_stats(const float* a, const float* b, int B, int H, int W,
                    float* cavg, float* cmax,        // [B,H,W]
                    float* havg, float* hmax,        // [B,C,W]  (reduced over H)
                    float* wavg, float* wmax,        // [B,H,C]  (reduced over W; row-major in y so that a band's halo rows are contiguous)
                    cudaStream_t st, int Hf = 0);
// top / bot (band mode): cavg, cmax, wavg, wmax carry one valid halo row above / below
int launch_ua_small_convs(int B, int H, int W, UaW w, const float* cavg, const float* cmax, const float* havg, const float* hmax,
                          const float* wavg, const float* wmax, float* c_att, float* h_att, float* w_att, cudaStream_t st, int top = 0, int bot = 0);
// out_sum / out_max [180] = sum / max over the nparts partials of one image (band mode: the vectors that are all-reduced)
int launch_reduce_parts(const float* part_sum, const float* part_max, int nparts, float* out_sum, float* out_max, cudaStream_t st);
// S[n, c] = c_att[y,x] + w_att[c,y] + h_att[c,x]  -> bf16 [N,192]
int launch_ua_build(int B, int H, int W, const float* c_att, const float* h_att, const float* w_att, bf16* s, cudaStream_t st);
// out = first*sigmoid(a1*sigmoid(a2)) + second*sigmoid(a3*(1-sigmoid(a2)))  -> bf16 [N,192] (+ fp32 tap)
int launch_fusion_combine(const float* first, const float* second, const float* a1, const float* a2, const float* a3,
                          bf16* out, float* out_f32, long long N, cudaStream_t st);

// ---- pack.cu (weight-only precomputation) --------------------------------------------------------
// conv / linear weight fp32 [Co][Ci][kh][kw] -> bf16 [Npad][taps*Cipad], k = tap*Cipad + ci; bias -> fp32 [Npad]
// perm_k != 0 (linear only): K index = head-padded position, i.e. wp[n][p] = w[n][scc_chan(p)]
int launch_pack_subpixel(const float* w, const float* b, bf16* wp, float* bp, cudaStream_t st);   // [64][64][3][3] -> four 2x2 phase filters [64][16*64]
int launch_pack_fold_last(const float* w, bf16* wp, int Co, cudaStream_t st);   // [Co<=4][64][3][3] -> [48][64], row = tap * 4 + co
int launch_pack_conv(const float* w, const float* b, bf16* wp, float* bp, int Co, int Ci, int taps, int Npad, int Cipad, int perm_k, cudaStream_t st);
// MultipleSizeConvExtract: conv3/5/7/9 + conv_x embedded in a 9x9x3 footprint, rows grouped per 32 channels x 5 responses (EPI_MSGATE)
int launch_pack_msconv(const float* w3, const float* w5, const float* w7, const float* w9, const float* wx,
                       const float* b3, const float* b5, const float* b7, const float* b9, const float* bx,
                       bf16* wp, float* bp, int in_ch, int Kp, cudaStream_t st);
// conv_first.conv_last for the [tile][slot][32 ch] order of the gated concat (EPI_MSGATE output)
int launch_pack_mslast(const float* w, const float* b, bf16* wp, float* bp, int Npad, cudaStream_t st);
// first-layer plain conv (f x f footprint over in_ch) -> [192][Kp] with k = (ky*f+kx)*in_ch + ci
int launch_pack_firstconv(const float* w, const float* b, bf16* wp, float* bp, int Co, int in_ch, int f, int Kp, cudaStream_t st);
// [C][1][kh][kw] -> [kh*kw][Cpad] fp32 (tap major); used for depthwise 5x5 (C=360->384) and casa 3x3 (1->C)
int launch_pack_tapmajor(const float* w, float* out, int C, int taps, int Cpad, cudaStream_t st);
struct PosW {
  const float* proj_w; const float* proj_b;   // [11][2], [11]
  const float* ln_w[3]; const float* ln_b[3]; // [11] x3
  const float* fc_w[3]; const float* fc_b[3]; // [11][11],[11][11],[6][11]
};
// DynamicPosBias MLP over all (2w-1)^2 offsets -> tbl [(2w-1)^2][6]; then pooled bias [6][L][Lb]
int launch_pos_table(PosW w, int win, float* tbl, cudaStream_t st);
int launch_pooled_bias(const float* tbl, int win, int base, float* out, cudaStream_t st);

}  // namespace hitsir
