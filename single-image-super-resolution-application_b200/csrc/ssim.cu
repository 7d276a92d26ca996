// Y-channel SSIM on the device (hitsir_ssim_y): skimage 0.24's structural_similarity(hr_y, sr_y, data_range=1) of every image of two
// fp32 NCHW [B,3,H,W] batches, the second metric of the reference evaluation (experiments/experiment.py:575-640) next to psnr_y.
//
// One CTA computes a 32 x 32 tile of the SSIM map's interior [R, H-R) x [R, W-R), R = window radius, whose windows all lie inside the
// image.  It stages the tile plus an R-pixel halo as two fp32 Y tiles in shared memory (y_channel, ycbcr.cuh), runs the horizontal pass
// of the five window moments (x, y, x*x, y*y, x*y; products rounded to fp32 as numpy forms them) into shared memory as doubles, then
// the vertical pass.  The window sums are accumulated in double and rounded to fp32 once, so each moment carries one fp32 rounding
// (scipy's filters round after each of the two passes); the SSIM formula after it is skimage's fp32 expression, operation by
// operation, with explicit _rn intrinsics, which makes ssim(x, x) exactly 1.  S is summed in double per thread, then thread -> warp
// -> CTA in a fixed order into partial[b][tile]; ssim_y_final_kernel sums an image's tiles in a fixed order.  No atomics: the result
// is bitwise reproducible and an image's value does not depend on the rest of the batch.
//
// The second half of the file scores by BasicSR's convention instead (hitsir_psnr_ssim_basicsr): uint8 inputs, crop_border, BasicSR's
// Y or the colour channels, and float64 throughout, with the same tile geometry and fixed-order reductions.
#include <cmath>
#include <type_traits>

#include "kernels.cuh"
#include "ycbcr.cuh"

namespace hitsir {
namespace {

constexpr int kSsimTile = 32;          // output pixels per tile side
constexpr int kSsimThreads = 256;
constexpr int kMaxTaps = 11;

struct SsimWin {
  double w[kMaxTaps];   // 1-D taps: 1 (uniform) or scipy's _gaussian_kernel1d(sigma = 1.5, radius 5)
  double scale;         // applied to the 2-D window sum: 1 / win^2 (uniform) or 1 (the Gaussian taps are normalised)
  float cn;             // covariance normalisation win^2 / (win^2 - 1) or 1, fp32 as numpy applies the Python float
};

template <int R>
constexpr size_t ssim_smem_bytes() {
  return (size_t)5 * (kSsimTile + 2 * R) * kSsimTile * sizeof(double) + (size_t)2 * (kSsimTile + 2 * R) * (kSsimTile + 2 * R) * sizeof(float);
}

template <int R>
__global__ void __launch_bounds__(kSsimThreads) ssim_y_partial_kernel(const float* __restrict__ sr, const float* __restrict__ hr, int H, int W,
                                                                      int clip, SsimWin win, int tiles_x, double* __restrict__ partial) {
  constexpr int T = kSsimTile, N = T + 2 * R, K = 2 * R + 1;
  extern __shared__ __align__(16) unsigned char smem[];
  double* hs = reinterpret_cast<double*>(smem);          // [5][N rows][T cols]: horizontal window sums
  float* sx = reinterpret_cast<float*>(hs + 5 * N * T);  // [N][N] Y of hr (skimage's im1)
  float* sy = sx + N * N;                                // [N][N] Y of sr (im2)
  __shared__ double s_w[kSsimThreads / 32];

  const int b = blockIdx.y, tile = blockIdx.x;
  const int ty = tile / tiles_x, tx = tile - ty * tiles_x;
  const int oy0 = R + ty * T, ox0 = R + tx * T;          // first output pixel of the tile; its staged region starts R rows / cols above
  const long long HW = (long long)H * W;
  const float* s0 = sr + (long long)b * 3 * HW;
  const float* h0 = hr + (long long)b * 3 * HW;

  for (int i = threadIdx.x; i < N * N; i += kSsimThreads) {
    const int r = i / N, c = i - r * N;
    // a partial last tile clamps its loads; the clamped pixels only feed outputs that are not summed
    const long long px = (long long)min(oy0 - R + r, H - 1) * W + min(ox0 - R + c, W - 1);
    float rr = s0[px], g = s0[HW + px], bl = s0[2 * HW + px];
    if (clip) { rr = fminf(fmaxf(rr, 0.f), 1.f); g = fminf(fmaxf(g, 0.f), 1.f); bl = fminf(fmaxf(bl, 0.f), 1.f); }
    sy[i] = y_channel(rr, g, bl);
    sx[i] = y_channel(h0[px], h0[HW + px], h0[2 * HW + px]);
  }
  __syncthreads();

  for (int i = threadIdx.x; i < N * T; i += kSsimThreads) {
    const int r = i / T, c = i - r * T;
    const float* px = sx + r * N + c;
    const float* py = sy + r * N + c;
    double m0 = 0.0, m1 = 0.0, m2 = 0.0, m3 = 0.0, m4 = 0.0;
#pragma unroll
    for (int j = 0; j < K; ++j) {
      const double w = win.w[j];
      const float xv = px[j], yv = py[j];
      m0 = fma(w, (double)xv, m0);
      m1 = fma(w, (double)yv, m1);
      m2 = fma(w, (double)__fmul_rn(xv, xv), m2);
      m3 = fma(w, (double)__fmul_rn(yv, yv), m3);
      m4 = fma(w, (double)__fmul_rn(xv, yv), m4);
    }
    hs[(0 * N + r) * T + c] = m0;
    hs[(1 * N + r) * T + c] = m1;
    hs[(2 * N + r) * T + c] = m2;
    hs[(3 * N + r) * T + c] = m3;
    hs[(4 * N + r) * T + c] = m4;
  }
  __syncthreads();

  const float C1 = (float)(0.01 * 0.01), C2 = (float)(0.03 * 0.03), cn = win.cn;
  const int ny = min(T, H - R - oy0), nx = min(T, W - R - ox0);
  double acc = 0.0;
  for (int i = threadIdx.x; i < T * T; i += kSsimThreads) {
    const int r = i / T, c = i - r * T;
    if (r >= ny || c >= nx) continue;
    double m0 = 0.0, m1 = 0.0, m2 = 0.0, m3 = 0.0, m4 = 0.0;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const double w = win.w[k];
      m0 = fma(w, hs[(0 * N + r + k) * T + c], m0);
      m1 = fma(w, hs[(1 * N + r + k) * T + c], m1);
      m2 = fma(w, hs[(2 * N + r + k) * T + c], m2);
      m3 = fma(w, hs[(3 * N + r + k) * T + c], m3);
      m4 = fma(w, hs[(4 * N + r + k) * T + c], m4);
    }
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
    acc += (double)__fdiv_rn(__fmul_rn(A1, A2), __fmul_rn(B1, B2));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < kSsimThreads / 32; ++w) t += s_w[w];
    partial[(long long)b * gridDim.x + tile] = t;
  }
}

// one warp: lane l sums p[l], p[l+32], ... in order, then a butterfly (every lane ends with the same, order-fixed value)
__device__ __forceinline__ double warp_fixed_sum(const double* __restrict__ p, int n) {
  double t = 0.0;
  for (int c = threadIdx.x; c < n; c += 32) t += p[c];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
  return t;
}

// one warp per image
__global__ void ssim_y_final_kernel(const double* __restrict__ partial, int tiles, double count, double* __restrict__ ssim) {
  const double t = warp_fixed_sum(partial + (long long)blockIdx.x * tiles, tiles);
  if (threadIdx.x == 0) ssim[blockIdx.x] = t / count;
}

template <int R>
int launch_partial(const float* sr, const float* hr, int B, int H, int W, int clip, const SsimWin& win, int tiles_x, int tiles, double* partial,
                   cudaStream_t st) {
  constexpr size_t smem = ssim_smem_bytes<R>();
  HITSIR_CHECK(cudaFuncSetAttribute(ssim_y_partial_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  ssim_y_partial_kernel<R><<<dim3((unsigned)tiles, (unsigned)B), kSsimThreads, smem, st>>>(sr, hr, H, W, clip, win, tiles_x, partial);
  HITSIR_CHECK(cudaGetLastError());
  return 0;
}

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

constexpr size_t bsr_smem_bytes() {
  return (size_t)5 * (kSsimTile + 2 * kBsrR) * kSsimTile * sizeof(double) + (size_t)2 * (kSsimTile + 2 * kBsrR) * (kSsimTile + 2 * kBsrR) * sizeof(double);
}

template <bool Y>
__device__ __forceinline__ double bsr_value(const uint8_t* px, int plane) {
  return Y ? (double)y_basicsr(px[0], px[1], px[2]) : (double)px[plane];
}

// One CTA per 32 x 32 tile of the valid region of plane blockIdx.y of image blockIdx.z.  Stages the tile plus a 5-pixel halo as
// doubles, runs the horizontal then the vertical 11-tap pass of the five moments in double (the products are exact: fp32 x fp32 or
// integers), evaluates BasicSR's ssim_map expression operation by operation (so ssim(x, x) is exactly 1: with img == img2 the numerator
// and denominator factors are equal bitwise), and reduces thread -> warp -> CTA in a fixed order into partial[b][plane][tile].
template <bool Y>
__global__ void __launch_bounds__(kSsimThreads) basicsr_ssim_partial_kernel(const uint8_t* __restrict__ sr, const uint8_t* __restrict__ hr, int H,
                                                                            int W, int crop, int tiles_x, double* __restrict__ partial) {
  constexpr int T = kSsimTile, R = kBsrR, N = T + 2 * R, K = 2 * R + 1;
  extern __shared__ __align__(16) unsigned char smem[];
  double* hs = reinterpret_cast<double*>(smem);   // [5][N rows][T cols]: horizontal window sums
  double* sa = hs + 5 * N * T;                    // [N][N] sr plane (BasicSR's img)
  double* sb = sa + N * N;                        // [N][N] hr plane (img2)
  __shared__ double s_w[kSsimThreads / 32];

  const int tile = blockIdx.x, plane = blockIdx.y, b = blockIdx.z;
  const int ty = tile / tiles_x, tx = tile - ty * tiles_x;
  const int oy0 = crop + R + ty * T, ox0 = crop + R + tx * T;
  const uint8_t* s0 = sr + (long long)b * H * W * 3;
  const uint8_t* h0 = hr + (long long)b * H * W * 3;

  for (int i = threadIdx.x; i < N * N; i += kSsimThreads) {
    const int r = i / N, c = i - r * N;
    // a partial last tile clamps its loads; the clamped pixels only feed outputs that are not summed
    const long long px = ((long long)min(oy0 - R + r, H - 1) * W + min(ox0 - R + c, W - 1)) * 3;
    sa[i] = bsr_value<Y>(s0 + px, plane);
    sb[i] = bsr_value<Y>(h0 + px, plane);
  }
  __syncthreads();

  for (int i = threadIdx.x; i < N * T; i += kSsimThreads) {
    const int r = i / T, c = i - r * T;
    const double* pa = sa + r * N + c;
    const double* pb = sb + r * N + c;
    double m0 = 0.0, m1 = 0.0, m2 = 0.0, m3 = 0.0, m4 = 0.0;
#pragma unroll
    for (int j = 0; j < K; ++j) {
      const double w = kBsrGauss[j], a = pa[j], v = pb[j];
      m0 = fma(w, a, m0);
      m1 = fma(w, v, m1);
      m2 = fma(w, __dmul_rn(a, a), m2);
      m3 = fma(w, __dmul_rn(v, v), m3);
      m4 = fma(w, __dmul_rn(a, v), m4);
    }
    hs[(0 * N + r) * T + c] = m0;
    hs[(1 * N + r) * T + c] = m1;
    hs[(2 * N + r) * T + c] = m2;
    hs[(3 * N + r) * T + c] = m3;
    hs[(4 * N + r) * T + c] = m4;
  }
  __syncthreads();

  const double c1 = (0.01 * 255) * (0.01 * 255), c2 = (0.03 * 255) * (0.03 * 255);   // BasicSR's (0.01 * 255)**2, (0.03 * 255)**2
  const int ny = min(T, H - crop - R - oy0), nx = min(T, W - crop - R - ox0);
  double acc = 0.0;
  for (int i = threadIdx.x; i < T * T; i += kSsimThreads) {
    const int r = i / T, c = i - r * T;
    if (r >= ny || c >= nx) continue;
    double mu1 = 0.0, mu2 = 0.0, e11 = 0.0, e22 = 0.0, e12 = 0.0;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const double w = kBsrGauss[k];
      mu1 = fma(w, hs[(0 * N + r + k) * T + c], mu1);
      mu2 = fma(w, hs[(1 * N + r + k) * T + c], mu2);
      e11 = fma(w, hs[(2 * N + r + k) * T + c], e11);
      e22 = fma(w, hs[(3 * N + r + k) * T + c], e22);
      e12 = fma(w, hs[(4 * N + r + k) * T + c], e12);
    }
    const double mu1_sq = __dmul_rn(mu1, mu1), mu2_sq = __dmul_rn(mu2, mu2), mu1_mu2 = __dmul_rn(mu1, mu2);
    const double s1 = __dsub_rn(e11, mu1_sq), s2 = __dsub_rn(e22, mu2_sq), s12 = __dsub_rn(e12, mu1_mu2);
    const double num = __dmul_rn(__dadd_rn(__dmul_rn(2.0, mu1_mu2), c1), __dadd_rn(__dmul_rn(2.0, s12), c2));
    const double den = __dmul_rn(__dadd_rn(__dadd_rn(mu1_sq, mu2_sq), c1), __dadd_rn(__dadd_rn(s1, s2), c2));
    acc = __dadd_rn(acc, __ddiv_rn(num, den));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < kSsimThreads / 32; ++w) t += s_w[w];
    partial[((long long)b * gridDim.y + plane) * gridDim.x + tile] = t;
  }
}

// Sum of squared differences over the crop [c, H-c) x [c, W-c) of image blockIdx.y, kBsrChunk pixels per CTA.  Y: the fp32 Y values'
// difference (exact in double) squared and summed in double in a fixed order.  RGB: the integer differences of all three channels,
// summed exactly in int64; a CTA's sum stays far below 2^53, so the partials and their sum are exact doubles and the MSE equals numpy's.
template <bool Y>
__global__ void __launch_bounds__(256) basicsr_sse_partial_kernel(const uint8_t* __restrict__ sr, const uint8_t* __restrict__ hr, int H, int W,
                                                                  int crop, double* __restrict__ partial) {
  using Acc = typename std::conditional<Y, double, long long>::type;
  __shared__ Acc s_w[8];
  const int b = blockIdx.y, Wc = W - 2 * crop;
  const long long n = (long long)(H - 2 * crop) * Wc;
  const uint8_t* s0 = sr + (long long)b * H * W * 3;
  const uint8_t* h0 = hr + (long long)b * H * W * 3;
  Acc acc = 0;
  const long long base = (long long)blockIdx.x * kBsrChunk;
#pragma unroll 4
  for (int i = 0; i < kBsrChunk / 256; ++i) {
    const long long p = base + threadIdx.x + 256 * i;
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
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    Acc t = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += s_w[w];
    partial[(long long)b * gridDim.x + blockIdx.x] = (double)t;
  }
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
  constexpr size_t smem = bsr_smem_bytes();
  double* ssim_partial = scratch;
  double* sse_partial = scratch + (long long)B * planes * tiles;
  HITSIR_CHECK(cudaFuncSetAttribute(basicsr_ssim_partial_kernel<Y>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  basicsr_ssim_partial_kernel<Y><<<dim3((unsigned)tiles, planes, (unsigned)B), kSsimThreads, smem, st>>>(sr, hr, H, W, crop, tiles_x, ssim_partial);
  HITSIR_CHECK(cudaGetLastError());
  basicsr_sse_partial_kernel<Y><<<dim3((unsigned)chunks, (unsigned)B), 256, 0, st>>>(sr, hr, H, W, crop, sse_partial);
  HITSIR_CHECK(cudaGetLastError());
  const double count = (double)(H - 2 * crop - 2 * kBsrR) * (double)(W - 2 * crop - 2 * kBsrR);
  basicsr_final_kernel<<<B, 32, 0, st>>>(ssim_partial, tiles, planes, count, sse_partial, chunks,
                                         (double)(H - 2 * crop) * (double)(W - 2 * crop) * (Y ? 1.0 : 3.0), mse, ssim);
  HITSIR_CHECK(cudaGetLastError());
  return 0;
}

}  // namespace

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
  const int rc = gaussian ? launch_partial<5>(sr, hr, B, H, W, clip, win, tiles_x, (int)tiles, partial, st)
                          : launch_partial<3>(sr, hr, B, H, W, clip, win, tiles_x, (int)tiles, partial, st);
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
