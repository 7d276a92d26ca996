// Evaluation metrics on the device, per image of two batches:
//  * psnr_y (hitsir_psnr_y): the Y-channel MSE of two [0,1] fp32 NCHW [B,3,H,W] batches, the first metric of the reference evaluation
//    (experiments/experiment.py:436-463);
//  * ssim_y (hitsir_ssim_y): skimage 0.24's structural_similarity(hr_y, sr_y, data_range=1) of the same batches, the second metric
//    (experiments/experiment.py:575-640);
//  * psnr_ssim_basicsr (hitsir_psnr_ssim_basicsr): the same two scores by BasicSR's convention instead: uint8 inputs, crop_border,
//    BasicSR's Y or the colour channels, and float64 throughout.
// Both SSIMs run one tile kernel (ssim_tile_kernel); a convention struct (SkimageY, BasicsrPlane) supplies what differs.  Every partial
// kernel reduces its CTA through block_fixed_sum and every final kernel sums an image's partials in a fixed order.  No atomics: the
// results are bitwise reproducible and an image's value does not depend on the rest of the batch.
#include <cmath>
#include <type_traits>

#include "kernels.cuh"
#include "ycbcr.cuh"

namespace hitsir {
namespace {

constexpr int kThreads = 256;          // threads of every partial kernel: the 8 warps block_fixed_sum adds
constexpr int kSsimTile = 32;          // output pixels per tile side
constexpr int kMaxTaps = 11;

// Sum of v over the CTA in a fixed order: a xor butterfly within each warp, lane 0 of each warp stores, then thread 0 adds the warp sums
// 0..7 in order.  The sum is returned to thread 0 only.
template <typename T>
__device__ __forceinline__ T block_fixed_sum(T v) {
  __shared__ T s_w[kThreads / 32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = v;
  __syncthreads();
  T t = 0;
  if (threadIdx.x == 0) {
#pragma unroll
    for (int w = 0; w < kThreads / 32; ++w) t += s_w[w];
  }
  return t;
}

// one warp: lane l sums p[l], p[l+32], ... in order, then a butterfly (every lane ends with the same, order-fixed value)
__device__ __forceinline__ double warp_fixed_sum(const double* __restrict__ p, int n) {
  double t = 0.0;
  for (int c = threadIdx.x; c < n; c += 32) t += p[c];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
  return t;
}

// psnr_y: Y channel of both [0,1] RGB batches exactly as utils/utils.py:170-186 writes it (y_channel, ycbcr.cuh), then the squared fp32
// difference accumulated in double (skimage mean_squared_error: float32 squares, float64 mean).  Two fixed-order levels (thread -> warp
// tree -> CTA partial -> per-image sum).
constexpr int kPsnrChunk = 4096;                           // pixels per CTA
__global__ void __launch_bounds__(kThreads) psnr_y_partial_kernel(const float* __restrict__ sr, const float* __restrict__ hr, long long HW, int clip,
                                                                  double* __restrict__ partial) {
  const int b = blockIdx.y;
  const float* s0 = sr + (long long)b * 3 * HW;
  const float* h0 = hr + (long long)b * 3 * HW;
  double acc = 0.0;
  const long long base = (long long)blockIdx.x * kPsnrChunk;
#pragma unroll 4
  for (int i = 0; i < kPsnrChunk / kThreads; ++i) {
    const long long px = base + threadIdx.x + kThreads * i;
    if (px < HW) {
      float r = s0[px], g = s0[HW + px], bl = s0[2 * HW + px];
      if (clip) { r = fminf(fmaxf(r, 0.f), 1.f); g = fminf(fmaxf(g, 0.f), 1.f); bl = fminf(fmaxf(bl, 0.f), 1.f); }   // sr_imgs.clip(0, 1) (:748)
      const float d = __fsub_rn(y_channel(h0[px], h0[HW + px], h0[2 * HW + px]), y_channel(r, g, bl));
      acc += (double)__fmul_rn(d, d);
    }
  }
  const double t = block_fixed_sum(acc);
  if (threadIdx.x == 0) partial[(long long)b * gridDim.x + blockIdx.x] = t;
}
__global__ void psnr_y_final_kernel(const double* __restrict__ partial, int chunks, long long HW, double* __restrict__ mse) {
  if (threadIdx.x != 0) return;
  double t = 0.0;
  for (int c = 0; c < chunks; ++c) t += partial[(long long)blockIdx.x * chunks + c];
  mse[blockIdx.x] = t / (double)HW;
}

struct SsimWin {
  double w[kMaxTaps];   // 1-D taps: 1 (uniform) or scipy's _gaussian_kernel1d(sigma = 1.5, radius 5)
  double scale;         // applied to the 2-D window sum: 1 / win^2 (uniform) or 1 (the Gaussian taps are normalised)
  float cn;             // covariance normalisation win^2 / (win^2 - 1) or 1, fp32 as numpy applies the Python float
};

// A convention of ssim_tile_kernel supplies: R, the window radius; In, the input element type; Val, the staged type; load, the staged
// values x and y of a pixel of both images; tap(j), the 1-D window; sq(a, b), a product of two staged values as a double; score, S
// from the five window moments of x, y, x*x, y*y and x*y.

// skimage: x is the fp32 Y of hr (skimage's im1), y that of sr (im2), sr clipped to [0, 1] first when clip.  The products are rounded to
// fp32 as numpy forms them.  The window sums are accumulated in double and rounded to fp32 once, so each moment carries one fp32
// rounding (scipy's filters round after each of the two passes); the SSIM formula after it is skimage's fp32 expression, operation by
// operation, with explicit _rn intrinsics, which makes ssim(x, x) exactly 1.
template <int Radius>
struct SkimageY {
  static constexpr int R = Radius;
  using In = float;
  using Val = float;
  SsimWin win;
  int clip;

  __device__ __forceinline__ void load(const float* sr, const float* hr, long long HW, long long px, int, float& x, float& y) const {
    float rr = sr[px], g = sr[HW + px], bl = sr[2 * HW + px];
    if (clip) { rr = fminf(fmaxf(rr, 0.f), 1.f); g = fminf(fmaxf(g, 0.f), 1.f); bl = fminf(fmaxf(bl, 0.f), 1.f); }
    y = y_channel(rr, g, bl);
    x = y_channel(hr[px], hr[HW + px], hr[2 * HW + px]);
  }
  // The tap is read from a copy of the window: read in place from the kernel parameter, it made ptxas (CUDA 12.9) allocate 37
  // registers instead of 32 for R = 3.
  __device__ __forceinline__ double tap(int j) const {
    const SsimWin w = win;
    return w.w[j];
  }
  static __device__ __forceinline__ double sq(float a, float b) { return (double)__fmul_rn(a, b); }
  __device__ __forceinline__ double score(double m0, double m1, double m2, double m3, double m4) const {
    const float C1 = (float)(0.01 * 0.01), C2 = (float)(0.03 * 0.03), cn = win.cn;
    const float ux = __double2float_rn(m0 * win.scale), uy = __double2float_rn(m1 * win.scale);
    const float uxx = __double2float_rn(m2 * win.scale), uyy = __double2float_rn(m3 * win.scale), uxy = __double2float_rn(m4 * win.scale);
    // skimage: vx = cov_norm * (uxx - ux * ux), ...; A1, A2, B1, B2 = 2*ux*uy + C1, 2*vxy + C2, ux**2 + uy**2 + C1, vx + vy + C2;
    // S = (A1 * A2) / (B1 * B2).  With x == y: A1 == B1 and A2 == B2 bitwise (doubling is exact), so S == 1.
    const float vx = __fmul_rn(cn, __fsub_rn(uxx, __fmul_rn(ux, ux)));
    const float vy = __fmul_rn(cn, __fsub_rn(uyy, __fmul_rn(uy, uy)));
    const float vxy = __fmul_rn(cn, __fsub_rn(uxy, __fmul_rn(ux, uy)));
    const float A1 = __fadd_rn(__fmul_rn(__fmul_rn(2.f, ux), uy), C1);
    const float A2 = __fadd_rn(__fmul_rn(2.f, vxy), C2);
    const float B1 = __fadd_rn(__fadd_rn(__fmul_rn(ux, ux), __fmul_rn(uy, uy)), C1);
    const float B2 = __fadd_rn(__fadd_rn(vx, vy), C2);
    return (double)__fdiv_rn(__fmul_rn(A1, A2), __fmul_rn(B1, B2));
  }
};

// ---- BasicSR 1.4.2's calculate_psnr / calculate_ssim (basicsr/metrics/psnr_ssim.py) of two uint8 RGB HWC batches ----
//
// A plane is BasicSR's Y (y_basicsr, 0-255 scale) when Y, else one colour channel.  Everything after the plane values is float64, as
// BasicSR computes it.  The window is cv2.getGaussianKernel(11, 1.5), these exact doubles, applied as outer(k, k); only the "valid"
// region [c+5, H-c-5) x [c+5, W-c-5) of the crop is kept, as BasicSR's [5:-5, 5:-5] of filter2D does.
__constant__ double kBsrGauss[11] = {0x1.0d956b52a1d6ep-10, 0x1.f1fe01ae5a5b5p-8, 0x1.26eb175d83f66p-5, 0x1.bff0fe8e98418p-4,
                                     0x1.b43c3f52b19f3p-3,  0x1.106560aa892bfp-2, 0x1.b43c3f52b19f3p-3, 0x1.bff0fe8e98418p-4,
                                     0x1.26eb175d83f66p-5,  0x1.f1fe01ae5a5b5p-8, 0x1.0d956b52a1d6ep-10};
constexpr int kBsrR = 5;
constexpr int kBsrChunk = 4096;        // cropped pixels per CTA of the squared-difference pass

// BasicSR's SSIM of one plane: x is the plane of sr (BasicSR's img), y that of hr (img2), staged as doubles.  The products are exact
// (fp32 x fp32 or integers).  S is BasicSR's ssim_map expression operation by operation, so ssim(x, x) is exactly 1: with img == img2
// the numerator and denominator factors are equal bitwise.
template <bool Y>
struct BasicsrPlane {
  static constexpr int R = kBsrR;
  using In = uint8_t;
  using Val = double;

  static __device__ __forceinline__ double value(const uint8_t* px, int plane) {
    return Y ? (double)y_basicsr(px[0], px[1], px[2]) : (double)px[plane];
  }
  __device__ __forceinline__ void load(const uint8_t* sr, const uint8_t* hr, long long, long long px, int plane, double& x, double& y) const {
    x = value(sr + px * 3, plane);
    y = value(hr + px * 3, plane);
  }
  __device__ __forceinline__ double tap(int j) const { return kBsrGauss[j]; }
  static __device__ __forceinline__ double sq(double a, double b) { return __dmul_rn(a, b); }
  __device__ __forceinline__ double score(double mu1, double mu2, double e11, double e22, double e12) const {
    const double c1 = (0.01 * 255) * (0.01 * 255), c2 = (0.03 * 255) * (0.03 * 255);   // BasicSR's (0.01 * 255)**2, (0.03 * 255)**2
    const double mu1_sq = __dmul_rn(mu1, mu1), mu2_sq = __dmul_rn(mu2, mu2), mu1_mu2 = __dmul_rn(mu1, mu2);
    const double s1 = __dsub_rn(e11, mu1_sq), s2 = __dsub_rn(e22, mu2_sq), s12 = __dsub_rn(e12, mu1_mu2);
    const double num = __dmul_rn(__dadd_rn(__dmul_rn(2.0, mu1_mu2), c1), __dadd_rn(__dmul_rn(2.0, s12), c2));
    const double den = __dmul_rn(__dadd_rn(__dadd_rn(mu1_sq, mu2_sq), c1), __dadd_rn(__dadd_rn(s1, s2), c2));
    return __ddiv_rn(num, den);
  }
};

template <class Conv>
constexpr size_t ssim_smem_bytes() {
  constexpr int N = kSsimTile + 2 * Conv::R;
  return (size_t)5 * N * kSsimTile * sizeof(double) + (size_t)2 * N * N * sizeof(typename Conv::Val);
}

// One CTA computes a 32 x 32 tile of the SSIM map of plane blockIdx.y of image blockIdx.z.  The map covers [c+R, H-c-R) x [c+R, W-c-R)
// of the crop c, R = window radius, whose windows all lie inside the crop (skimage: c = 0, the image's interior).  The CTA stages the
// tile plus an R-pixel halo of both images in shared memory, runs the horizontal pass of the five window moments into shared memory as
// doubles, then the vertical pass, and sums S in double per thread, then thread -> warp -> CTA in a fixed order into
// partial[b][plane][tile].
template <class Conv>
__global__ void __launch_bounds__(kThreads) ssim_tile_kernel(const typename Conv::In* __restrict__ sr, const typename Conv::In* __restrict__ hr,
                                                             int H, int W, int crop, int tiles_x, Conv conv, double* __restrict__ partial) {
  using Val = typename Conv::Val;
  constexpr int T = kSsimTile, R = Conv::R, N = T + 2 * R, K = 2 * R + 1;
  extern __shared__ __align__(16) unsigned char smem[];
  double* hs = reinterpret_cast<double*>(smem);      // [5][N rows][T cols]: horizontal window sums
  Val* sx = reinterpret_cast<Val*>(hs + 5 * N * T);  // [N][N] x
  Val* sy = sx + N * N;                              // [N][N] y

  const int tile = blockIdx.x, plane = blockIdx.y, b = blockIdx.z;
  const int ty = tile / tiles_x, tx = tile - ty * tiles_x;
  const int oy0 = crop + R + ty * T, ox0 = crop + R + tx * T;   // first output pixel of the tile; its staged region starts R rows / cols above
  const long long HW = (long long)H * W;
  const typename Conv::In* s0 = sr + (long long)b * 3 * HW;
  const typename Conv::In* h0 = hr + (long long)b * 3 * HW;

  for (int i = threadIdx.x; i < N * N; i += kThreads) {
    const int r = i / N, c = i - r * N;
    // a partial last tile clamps its loads; the clamped pixels only feed outputs that are not summed
    const long long px = (long long)min(oy0 - R + r, H - 1) * W + min(ox0 - R + c, W - 1);
    conv.load(s0, h0, HW, px, plane, sx[i], sy[i]);
  }
  __syncthreads();

  for (int i = threadIdx.x; i < N * T; i += kThreads) {
    const int r = i / T, c = i - r * T;
    const Val* px = sx + r * N + c;
    const Val* py = sy + r * N + c;
    double m0 = 0.0, m1 = 0.0, m2 = 0.0, m3 = 0.0, m4 = 0.0;
#pragma unroll
    for (int j = 0; j < K; ++j) {
      const double w = conv.tap(j);
      const Val xv = px[j], yv = py[j];
      m0 = fma(w, (double)xv, m0);
      m1 = fma(w, (double)yv, m1);
      m2 = fma(w, Conv::sq(xv, xv), m2);
      m3 = fma(w, Conv::sq(yv, yv), m3);
      m4 = fma(w, Conv::sq(xv, yv), m4);
    }
    hs[(0 * N + r) * T + c] = m0;
    hs[(1 * N + r) * T + c] = m1;
    hs[(2 * N + r) * T + c] = m2;
    hs[(3 * N + r) * T + c] = m3;
    hs[(4 * N + r) * T + c] = m4;
  }
  __syncthreads();

  const int ny = min(T, H - crop - R - oy0), nx = min(T, W - crop - R - ox0);
  double acc = 0.0;
  for (int i = threadIdx.x; i < T * T; i += kThreads) {
    const int r = i / T, c = i - r * T;
    if (r >= ny || c >= nx) continue;
    double m0 = 0.0, m1 = 0.0, m2 = 0.0, m3 = 0.0, m4 = 0.0;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const double w = conv.tap(k);
      m0 = fma(w, hs[(0 * N + r + k) * T + c], m0);
      m1 = fma(w, hs[(1 * N + r + k) * T + c], m1);
      m2 = fma(w, hs[(2 * N + r + k) * T + c], m2);
      m3 = fma(w, hs[(3 * N + r + k) * T + c], m3);
      m4 = fma(w, hs[(4 * N + r + k) * T + c], m4);
    }
    acc = __dadd_rn(acc, conv.score(m0, m1, m2, m3, m4));
  }
  const double t = block_fixed_sum(acc);
  if (threadIdx.x == 0) partial[((long long)b * gridDim.y + plane) * gridDim.x + tile] = t;
}

// grid (tiles, planes, B)
template <class Conv>
int launch_ssim_tiles(const typename Conv::In* sr, const typename Conv::In* hr, int B, int planes, int H, int W, int crop, int tiles_x, int tiles,
                      const Conv& conv, double* partial, cudaStream_t st) {
  constexpr size_t smem = ssim_smem_bytes<Conv>();
  HITSIR_CHECK(cudaFuncSetAttribute(ssim_tile_kernel<Conv>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  ssim_tile_kernel<Conv><<<dim3((unsigned)tiles, (unsigned)planes, (unsigned)B), kThreads, smem, st>>>(sr, hr, H, W, crop, tiles_x, conv, partial);
  HITSIR_CHECK(cudaGetLastError());
  return 0;
}

// one warp per image
__global__ void ssim_y_final_kernel(const double* __restrict__ partial, int tiles, double count, double* __restrict__ ssim) {
  const double t = warp_fixed_sum(partial + (long long)blockIdx.x * tiles, tiles);
  if (threadIdx.x == 0) ssim[blockIdx.x] = t / count;
}

// Sum of squared differences over the crop [c, H-c) x [c, W-c) of image blockIdx.y, kBsrChunk pixels per CTA.  Y: the fp32 Y values'
// difference (exact in double) squared and summed in double in a fixed order.  RGB: the integer differences of all three channels,
// summed exactly in int64; a CTA's sum stays far below 2^53, so the partials and their sum are exact doubles and the MSE equals numpy's.
template <bool Y>
__global__ void __launch_bounds__(kThreads) basicsr_sse_partial_kernel(const uint8_t* __restrict__ sr, const uint8_t* __restrict__ hr, int H, int W,
                                                                       int crop, double* __restrict__ partial) {
  using Acc = typename std::conditional<Y, double, long long>::type;
  const int b = blockIdx.y, Wc = W - 2 * crop;
  const long long n = (long long)(H - 2 * crop) * Wc;
  const uint8_t* s0 = sr + (long long)b * H * W * 3;
  const uint8_t* h0 = hr + (long long)b * H * W * 3;
  Acc acc = 0;
  const long long base = (long long)blockIdx.x * kBsrChunk;
#pragma unroll 4
  for (int i = 0; i < kBsrChunk / kThreads; ++i) {
    const long long p = base + threadIdx.x + kThreads * i;
    if (p < n) {
      const long long y = p / Wc, x = p - y * Wc;
      const long long px = ((y + crop) * W + x + crop) * 3;
      if constexpr (Y) {
        const double d = __dsub_rn((double)y_basicsr(s0[px], s0[px + 1], s0[px + 2]), (double)y_basicsr(h0[px], h0[px + 1], h0[px + 2]));
        acc = __dadd_rn(acc, __dmul_rn(d, d));
      } else {
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
          const long long d = (long long)s0[px + ch] - (long long)h0[px + ch];
          acc += d * d;
        }
      }
    }
  }
  const Acc t = block_fixed_sum(acc);
  if (threadIdx.x == 0) partial[(long long)b * gridDim.x + blockIdx.x] = (double)t;
}

// One warp per image: each plane's mean over the valid region; the channel mean as np.array(ssims).mean() forms it, ((B + G) + R) / 3
// (BasicSR's BGR order: our planes 2, 1, 0); and the MSE over the crop, sum / count as np.mean divides.
__global__ void basicsr_final_kernel(const double* __restrict__ ssim_partial, int tiles, int planes, double count, const double* __restrict__ sse_partial,
                                     int chunks, double n_sse, double* __restrict__ mse, double* __restrict__ ssim) {
  const int b = blockIdx.x;
  const double* p = ssim_partial + (long long)b * planes * tiles;
  double s = warp_fixed_sum(p, tiles) / count;
  if (planes == 3) s = ((warp_fixed_sum(p + 2LL * tiles, tiles) / count + warp_fixed_sum(p + tiles, tiles) / count) + s) / 3.0;
  const double sse = warp_fixed_sum(sse_partial + (long long)b * chunks, chunks);
  if (threadIdx.x == 0) {
    ssim[b] = s;
    mse[b] = sse / n_sse;
  }
}

template <bool Y>
int launch_basicsr(const uint8_t* sr, const uint8_t* hr, int B, int H, int W, int crop, int tiles_x, int tiles, int chunks, double* scratch,
                   double* mse, double* ssim, cudaStream_t st) {
  constexpr int planes = Y ? 1 : 3;
  double* ssim_partial = scratch;
  double* sse_partial = scratch + (long long)B * planes * tiles;
  if (launch_ssim_tiles(sr, hr, B, planes, H, W, crop, tiles_x, tiles, BasicsrPlane<Y>{}, ssim_partial, st)) return 1;
  basicsr_sse_partial_kernel<Y><<<dim3((unsigned)chunks, (unsigned)B), kThreads, 0, st>>>(sr, hr, H, W, crop, sse_partial);
  HITSIR_CHECK(cudaGetLastError());
  const double count = (double)(H - 2 * crop - 2 * kBsrR) * (double)(W - 2 * crop - 2 * kBsrR);
  basicsr_final_kernel<<<B, 32, 0, st>>>(ssim_partial, tiles, planes, count, sse_partial, chunks,
                                         (double)(H - 2 * crop) * (double)(W - 2 * crop) * (Y ? 1.0 : 3.0), mse, ssim);
  HITSIR_CHECK(cudaGetLastError());
  return 0;
}

}  // namespace

long long psnr_y_chunks(int H, int W) { return ((long long)H * W + kPsnrChunk - 1) / kPsnrChunk; }
int launch_psnr_y(const float* sr, const float* hr, int B, int H, int W, int clip, double* partial, double* mse, cudaStream_t st) {
  const long long HW = (long long)H * W, chunks = psnr_y_chunks(H, W);
  if (chunks > 2147483647LL || B > 65535) { set_error("launch_psnr_y: image or batch too large"); return 1; }
  psnr_y_partial_kernel<<<dim3((unsigned)chunks, (unsigned)B), kThreads, 0, st>>>(sr, hr, HW, clip, partial);
  HITSIR_CHECK(cudaGetLastError());
  psnr_y_final_kernel<<<B, 32, 0, st>>>(partial, (int)chunks, HW, mse);
  HITSIR_CHECK(cudaGetLastError());
  return 0;
}

int ssim_y_radius(int gaussian) { return gaussian ? 5 : 3; }   // uniform 7 x 7; Gaussian sigma 1.5, truncate 3.5: int(3.5 * 1.5 + 0.5)

long long ssim_y_tiles(int H, int W, int gaussian) {
  const int R = ssim_y_radius(gaussian);
  if (H < 2 * R + 1 || W < 2 * R + 1) return 0;
  return (long long)((H - 2 * R + kSsimTile - 1) / kSsimTile) * ((W - 2 * R + kSsimTile - 1) / kSsimTile);
}

int launch_ssim_y(const float* sr, const float* hr, int B, int H, int W, int clip, int gaussian, int sample_cov, double* partial, double* ssim,
                  cudaStream_t st) {
  const int R = ssim_y_radius(gaussian), K = 2 * R + 1;
  const long long tiles = ssim_y_tiles(H, W, gaussian);
  if (tiles == 0) { set_error("launch_ssim_y: image %d x %d is smaller than the %d x %d window", H, W, K, K); return 1; }
  if (tiles > 2147483647LL || B > 65535) { set_error("launch_ssim_y: image or batch too large"); return 1; }
  SsimWin win{};
  if (gaussian) {
    // scipy.ndimage._gaussian_kernel1d(sigma, 0, radius): phi = exp(-0.5 / sigma^2 * x^2), x = -R..R, phi / phi.sum()
    const double sigma = 1.5;
    double sum = 0.0;
    for (int j = 0; j < K; ++j) { win.w[j] = std::exp(-0.5 / (sigma * sigma) * (double)((j - R) * (j - R))); sum += win.w[j]; }
    for (int j = 0; j < K; ++j) win.w[j] /= sum;
    win.scale = 1.0;
  } else {
    for (int j = 0; j < K; ++j) win.w[j] = 1.0;
    win.scale = 1.0 / (double)(K * K);
  }
  win.cn = sample_cov ? (float)((double)(K * K) / (double)(K * K - 1)) : 1.0f;
  const int tiles_x = (W - 2 * R + kSsimTile - 1) / kSsimTile;
  const int rc = gaussian ? launch_ssim_tiles(sr, hr, B, 1, H, W, 0, tiles_x, (int)tiles, SkimageY<5>{win, clip}, partial, st)
                          : launch_ssim_tiles(sr, hr, B, 1, H, W, 0, tiles_x, (int)tiles, SkimageY<3>{win, clip}, partial, st);
  if (rc) return rc;
  ssim_y_final_kernel<<<B, 32, 0, st>>>(partial, (int)tiles, (double)(H - 2 * R) * (double)(W - 2 * R), ssim);
  HITSIR_CHECK(cudaGetLastError());
  return 0;
}

static long long basicsr_tiles(int H, int W, int crop) {
  const int vh = H - 2 * crop - 2 * kBsrR, vw = W - 2 * crop - 2 * kBsrR;
  return (long long)((vh + kSsimTile - 1) / kSsimTile) * ((vw + kSsimTile - 1) / kSsimTile);
}

static long long basicsr_chunks(int H, int W, int crop) {
  return ((long long)(H - 2 * crop) * (W - 2 * crop) + kBsrChunk - 1) / kBsrChunk;
}

int basicsr_metrics_check(int B, int H, int W, int crop) {
  if (B <= 0 || B > 65535 || crop < 0 || (long long)H - 2LL * crop < 2 * kBsrR + 1 || (long long)W - 2LL * crop < 2 * kBsrR + 1) {
    set_error("basicsr metrics: bad shape B=%d %d x %d with crop_border %d (B in 1..65535; H and W minus 2 * crop_border must be at least "
              "the 11 x 11 window)", B, H, W, crop);
    return 1;
  }
  if (basicsr_tiles(H, W, crop) > 2147483647LL || basicsr_chunks(H, W, crop) > 2147483647LL) { set_error("basicsr metrics: image too large"); return 1; }
  return 0;
}

long long basicsr_metrics_scratch_doubles(int B, int H, int W, int crop, int y_only) {
  return (long long)B * ((y_only ? 1 : 3) * basicsr_tiles(H, W, crop) + basicsr_chunks(H, W, crop));
}

int launch_psnr_ssim_basicsr(const uint8_t* sr, const uint8_t* hr, int B, int H, int W, int crop, int y_only, double* scratch, double* mse,
                             double* ssim, cudaStream_t st) {
  const int tiles_x = (W - 2 * crop - 2 * kBsrR + kSsimTile - 1) / kSsimTile;
  const int tiles = (int)basicsr_tiles(H, W, crop), chunks = (int)basicsr_chunks(H, W, crop);
  return y_only ? launch_basicsr<true>(sr, hr, B, H, W, crop, tiles_x, tiles, chunks, scratch, mse, ssim, st)
                : launch_basicsr<false>(sr, hr, B, H, W, crop, tiles_x, tiles, chunks, scratch, mse, ssim, st);
}

}  // namespace hitsir
