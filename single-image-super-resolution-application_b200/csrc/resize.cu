// Bicubic resizing on the device (hitsir_resize_u8_pil, hitsir_resize_f32_matlab): the LR synthesis of the reference evaluation
// (datasets/dataset.py:51-91) and the "Bicubic" baseline row, in two standard definitions that share one separable resampler.
//
// Tap tables.  For each output index o of an axis the table holds the first input index, the tap count and the weights, built on the
// device by resize_taps_kernel in the caller's scratch with explicitly rounded double operations (__dadd_rn / __dmul_rn / __ddiv_rn, no
// FMA contraction), so they equal a plain Python-float restatement bit for bit (tests/resize_ref.py) and the call needs no host copy.
//  * pil: Pillow 12.2 libImaging/Resample.c, precompute_coeffs + normalize_coeffs_8bpc: cubic a = -0.5, support 2 * max(in/out, 1),
//    weights normalised in double and converted to fixed point with 22 fractional bits.
//  * matlab: BasicSR's calculate_weights_indices (MATLAB imresize 'bicubic'): antialiased (width 4/scale) when downscaling, p =
//    ceil(width) + 2 taps starting at floor(u - width/2), half-sample symmetric boundary; fp64 weights rounded to fp32.  MATLAB drops the
//    all-zero first / last tap columns; they are kept here, since a zero weight adds an exact zero.
//
// Resampling.  One CTA computes a TH x TW output tile of one plane (an HWC image for pil, one channel of an NCHW image for matlab).  It
// stages the horizontal and vertical tap tables of the tile in shared memory, then walks the input rows the tile's vertical taps read in
// chunks of kRows: the horizontal pass writes a chunk's rows, restricted to the tile's output columns, into a shared-memory
// intermediate, and the vertical pass accumulates each output over the taps that fall into the chunk, in tap order.  The input itself is
// read by the horizontal pass through L1 instead of being staged: its column span grows with the downscale factor, the tables' only by
// the tap count.  pil: int32 sums from 1 << 21, clip8(sum >> 22), the intermediate uint8 exactly as Pillow's (horizontal pass first;
// Pillow restricts it to the rows the vertical pass reads, which changes no value).  matlab: fp32 FMA accumulation in tap order.
// No atomics: bitwise reproducible, and a plane's result does not depend on the rest of the batch.
#include <cmath>

#include "kernels.cuh"

namespace hitsir {
namespace {

constexpr int kThreads = 256;
constexpr int kTileH = 16;     // output rows per tile
constexpr int kRows = 80;      // intermediate rows per chunk: a x4 downscale of kTileH rows (4 * 16 + 12 taps) fits one chunk
constexpr int kPrecisionBits = 22;
constexpr int kMaxSmem = 227 * 1024;   // a CTA's shared memory on sm_100; the tap tables of a tile grow with the downscale factor

__host__ __device__ constexpr int tile_w(int ch) { return ch == 3 ? 32 : 64; }

// ---- tap tables ----------------------------------------------------------------------------------------------------------------------
// Pillow's bicubic_filter, operation by operation ((a+2) = 1.5, (a+3) = 2.5)
__device__ double pil_cubic(double x) {
  if (x < 0.0) x = -x;
  if (x < 1.0) return __dadd_rn(__dmul_rn(__dmul_rn(__dsub_rn(__dmul_rn(1.5, x), 2.5), x), x), 1.0);
  if (x < 2.0) return __dmul_rn(__dsub_rn(__dmul_rn(__dadd_rn(__dmul_rn(__dsub_rn(x, 5.0), x), 8.0), x), 4.0), -0.5);
  return 0.0;
}

// BasicSR's cubic: (1.5|x|^3 - 2.5|x|^2 + 1) on |x| <= 1, (-0.5|x|^3 + 2.5|x|^2 - 4|x| + 2) on 1 < |x| <= 2
__device__ double matlab_cubic(double x) {
  const double a = fabs(x), a2 = __dmul_rn(a, a), a3 = __dmul_rn(a2, a);
  if (a <= 1.0) return __dadd_rn(__dsub_rn(__dmul_rn(1.5, a3), __dmul_rn(2.5, a2)), 1.0);
  if (a <= 2.0) return __dadd_rn(__dsub_rn(__dadd_rn(__dmul_rn(-0.5, a3), __dmul_rn(2.5, a2)), __dmul_rn(4.0, a)), 2.0);
  return 0.0;
}

struct AxisSpec { int in, out, K; double scale; int* first; int* count; void* w; };

__device__ void pil_axis_row(const AxisSpec& a, int o) {
  const double scale = __ddiv_rn((double)a.in, (double)a.out);
  const double fs = scale < 1.0 ? 1.0 : scale;
  const double support = __dmul_rn(2.0, fs);
  const double center = __dmul_rn((double)o + 0.5, scale);
  const double ss = __ddiv_rn(1.0, fs);
  int xmin = __double2int_rz(__dadd_rn(__dsub_rn(center, support), 0.5));
  if (xmin < 0) xmin = 0;
  int xmax = __double2int_rz(__dadd_rn(__dadd_rn(center, support), 0.5));
  if (xmax > a.in) xmax = a.in;
  xmax -= xmin;
  double ww = 0.0;
  for (int x = 0; x < xmax; ++x) ww = __dadd_rn(ww, pil_cubic(__dmul_rn(__dadd_rn(__dsub_rn((double)(x + xmin), center), 0.5), ss)));
  int* w = static_cast<int*>(a.w) + (long long)o * a.K;
  for (int x = 0; x < xmax; ++x) {
    double k = pil_cubic(__dmul_rn(__dadd_rn(__dsub_rn((double)(x + xmin), center), 0.5), ss));
    if (ww != 0.0) k = __ddiv_rn(k, ww);
    const double f = __dmul_rn(k, (double)(1 << kPrecisionBits));
    w[x] = __double2int_rz(k < 0.0 ? __dadd_rn(-0.5, f) : __dadd_rn(0.5, f));
  }
  for (int x = xmax; x < a.K; ++x) w[x] = 0;
  a.first[o] = xmin;
  a.count[o] = xmax;
}

__device__ void matlab_axis_row(const AxisSpec& a, int o) {
  const double s = a.scale;
  const bool aa = s < 1.0;
  const double width = aa ? __ddiv_rn(4.0, s) : 4.0;
  const int p = (int)ceil(width) + 2;
  const double u = __dadd_rn(__ddiv_rn((double)(o + 1), s), __dmul_rn(0.5, __dsub_rn(1.0, __ddiv_rn(1.0, s))));
  const int left = (int)floor(__dsub_rn(u, __dmul_rn(width, 0.5)));     // 1-based index of tap 0
  double sum = 0.0;
  for (int k = 0; k < p; ++k) {
    const double d = __dsub_rn(u, (double)(left + k));
    sum = __dadd_rn(sum, aa ? __dmul_rn(s, matlab_cubic(__dmul_rn(d, s))) : matlab_cubic(d));
  }
  float* w = static_cast<float*>(a.w) + (long long)o * a.K;
  for (int k = 0; k < p; ++k) {
    const double d = __dsub_rn(u, (double)(left + k));
    w[k] = __double2float_rn(__ddiv_rn(aa ? __dmul_rn(s, matlab_cubic(__dmul_rn(d, s))) : matlab_cubic(d), sum));
  }
  a.first[o] = left - 1;
  a.count[o] = p;
}

// one thread per output index of both axes: [0, v.out) vertical, [v.out, v.out + h.out) horizontal
template <bool PIL>
__global__ void resize_taps_kernel(AxisSpec v, AxisSpec h) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= v.out + h.out) return;
  const AxisSpec& a = i < v.out ? v : h;
  const int o = i < v.out ? i : i - v.out;
  if (PIL) pil_axis_row(a, o);
  else matlab_axis_row(a, o);
}

// ---- resampling ----------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int mirror(int i, int n) {     // half-sample symmetric: ... 1 0 | 0 1 ... n-1 | n-1 n-2 ...
  if ((unsigned)i < (unsigned)n) return i;
  const int period = 2 * n;
  i %= period;
  if (i < 0) i += period;
  return i < n ? i : period - 1 - i;
}

__device__ __forceinline__ uint8_t clip8(int v) {           // Pillow's clip8 of a sum with kPrecisionBits fractional bits
  if (v >= (1 << kPrecisionBits << 8)) return 255;
  if (v <= 0) return 0;
  return (uint8_t)(v >> kPrecisionBits);
}

template <typename T> struct Acc;
template <> struct Acc<uint8_t> { typedef int W; typedef int A; };
template <> struct Acc<float> { typedef float W; typedef float A; };

struct Table { const int* first; const int* count; const void* w; int K; };

template <typename T, int CH>
size_t resize_smem_bytes(int Kv, int Kh) {
  constexpr int TW = tile_w(CH);
  return (size_t)kRows * TW * CH * sizeof(T) + 16 + (size_t)(2 * TW + TW * Kh + 2 * kTileH + kTileH * Kv) * 4;
}

template <typename T, int CH>
__global__ void __launch_bounds__(kThreads) resize_kernel(const T* __restrict__ src, T* __restrict__ dst, int H, int W, int outH, int outW,
                                                         Table tv, Table th) {
  typedef typename Acc<T>::W WT;
  typedef typename Acc<T>::A AT;
  constexpr bool kPil = sizeof(T) == 1;
  constexpr int TW = tile_w(CH), NCOL = TW * CH, NO = kTileH * NCOL / kThreads;
  static_assert(kTileH * NCOL % kThreads == 0, "outputs per thread");
  extern __shared__ __align__(16) unsigned char smem[];
  T* inter = reinterpret_cast<T*>(smem);                                      // [kRows][NCOL]
  int* hf = reinterpret_cast<int*>(smem + (((size_t)kRows * NCOL * sizeof(T) + 15) & ~(size_t)15));
  int* hc = hf + TW;
  WT* hw = reinterpret_cast<WT*>(hc + TW);                                    // [TW][Kh]
  int* vf = reinterpret_cast<int*>(hw + TW * th.K);
  int* vc = vf + kTileH;
  WT* vw = reinterpret_cast<WT*>(vc + kTileH);                                // [kTileH][Kv]

  const int ox0 = blockIdx.x * TW, oy0 = blockIdx.y * kTileH;
  const int nx = min(TW, outW - ox0), ny = min(kTileH, outH - oy0);
  const T* in = src + (long long)blockIdx.z * H * W * CH;
  T* out = dst + (long long)blockIdx.z * outH * outW * CH;

  for (int i = threadIdx.x; i < TW; i += kThreads) {
    hf[i] = i < nx ? th.first[ox0 + i] : 0;
    hc[i] = i < nx ? th.count[ox0 + i] : 0;
  }
  for (int i = threadIdx.x; i < kTileH; i += kThreads) {
    vf[i] = i < ny ? tv.first[oy0 + i] : 0;
    vc[i] = i < ny ? tv.count[oy0 + i] : 0;
  }
  for (int i = threadIdx.x; i < TW * th.K; i += kThreads) hw[i] = i < nx * th.K ? static_cast<const WT*>(th.w)[(long long)ox0 * th.K + i] : WT(0);
  for (int i = threadIdx.x; i < kTileH * tv.K; i += kThreads) vw[i] = i < ny * tv.K ? static_cast<const WT*>(tv.w)[(long long)oy0 * tv.K + i] : WT(0);
  __syncthreads();

  // both passes' first index and last end are non-decreasing in the output index
  const int ry0 = vf[0], ry1 = vf[ny - 1] + vc[ny - 1];
  AT acc[NO];
#pragma unroll
  for (int j = 0; j < NO; ++j) acc[j] = kPil ? AT(1 << (kPrecisionBits - 1)) : AT(0);

  for (int r0 = ry0; r0 < ry1; r0 += kRows) {
    const int n = min(kRows, ry1 - r0);
    for (int i = threadIdx.x; i < n * NCOL; i += kThreads) {
      const int rr = i / NCOL, col = i - rr * NCOL, x = col / CH, c = col - x * CH;
      const T* row = in + (long long)mirror(r0 + rr, H) * W * CH + c;
      const WT* w = hw + x * th.K;
      const int f = hf[x], cnt = hc[x];
      AT s = kPil ? AT(1 << (kPrecisionBits - 1)) : AT(0);
      for (int k = 0; k < cnt; ++k) {
        if constexpr (kPil) s += (int)row[(f + k) * CH] * w[k];
        else s = fmaf(w[k], row[(long long)mirror(f + k, W) * CH], s);
      }
      if constexpr (kPil) inter[i] = clip8(s);
      else inter[i] = s;
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < NO; ++j) {
      const int idx = threadIdx.x + j * kThreads, orow = idx / NCOL, col = idx - orow * NCOL;
      if (orow >= ny) continue;
      const int f = vf[orow], k0 = max(0, r0 - f), k1 = min(vc[orow], r0 + n - f);
      const WT* w = vw + orow * tv.K;
      for (int k = k0; k < k1; ++k) {
        if constexpr (kPil) acc[j] += (int)inter[(f + k - r0) * NCOL + col] * w[k];
        else acc[j] = fmaf(w[k], inter[(f + k - r0) * NCOL + col], acc[j]);
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int j = 0; j < NO; ++j) {
    const int idx = threadIdx.x + j * kThreads, orow = idx / NCOL, col = idx - orow * NCOL;
    if (orow >= ny || col >= nx * CH) continue;
    T* o = out + ((long long)(oy0 + orow) * outW + ox0) * CH + col;
    if constexpr (kPil) *o = clip8(acc[j]);
    else *o = acc[j];
  }
}

// scratch layout: first_v | count_v | w_v [outH][Kv] | first_h | count_h | w_h [outW][Kh], each region 256-byte aligned
size_t region(long long n) { return (size_t)((n * 4 + 255) / 256 * 256); }
size_t table_bytes(int out, int K) { return 2 * region(out) + region((long long)out * K); }

Table make_table(unsigned char* base, int out, int K, AxisSpec* spec, int in, double scale) {
  int* first = reinterpret_cast<int*>(base);
  int* count = reinterpret_cast<int*>(base + region(out));
  void* w = base + 2 * region(out);
  *spec = AxisSpec{in, out, K, scale, first, count, w};
  return Table{first, count, w, K};
}

template <typename T, int CH>
int launch_resample(const T* src, T* dst, int planes, int H, int W, int outH, int outW, const Table& tv, const Table& th, cudaStream_t st) {
  // the size varies from call to call: opt in to the largest once, resize_check keeps every launch within it
  static unsigned long long mask = 0;
  const size_t smem = resize_smem_bytes<T, CH>(tv.K, th.K);
  if (ensure_dynamic_smem(resize_kernel<T, CH>, kMaxSmem, &mask)) return 1;
  const dim3 grid((unsigned)cdiv(outW, tile_w(CH)), (unsigned)cdiv(outH, kTileH), (unsigned)planes);
  resize_kernel<T, CH><<<grid, kThreads, smem, st>>>(src, dst, H, W, outH, outW, tv, th);
  HITSIR_CHECK(cudaGetLastError());
  return 0;
}

template <bool PIL>
int launch_taps(const AxisSpec& v, const AxisSpec& h, cudaStream_t st) {
  const int n = v.out + h.out;
  resize_taps_kernel<PIL><<<cdiv(n, 128), 128, 0, st>>>(v, h);
  HITSIR_CHECK(cudaGetLastError());
  return 0;
}

}  // namespace

// Pillow's maximum tap count of an axis: (int)ceil(support) * 2 + 1, support = 2 * max(in / out, 1)
int resize_pil_taps(int in, int out) {
  const double scale = (double)in / (double)out;
  return (int)std::ceil(2.0 * (scale < 1.0 ? 1.0 : scale)) * 2 + 1;
}

// BasicSR's p = ceil(width) + 2 for `scale`, width = 4 / scale when downscaling
int resize_matlab_taps(double scale) { return (int)std::ceil(scale < 1.0 ? 4.0 / scale : 4.0) + 2; }

// An upper bound of resize_matlab_taps over every scale with ceil(in * scale) == out: scale > (out - 1) / in.  out == 1 bounds no
// scale from below; its tables are sized for scale >= 1 / max(in, 16).
int resize_matlab_taps_bound(int in, int out) {
  if (out < 2) return 4 * (in > 16 ? in : 16) + 2;
  const long long b = 4LL * in / (out - 1) + 3;
  return b < 6 ? 6 : (int)(b > (1 << 30) ? (1 << 30) : b);
}

int resize_check(int matlab, int C, int H, int W, int outH, int outW, double scale) {
  const int Kv = matlab ? resize_matlab_taps(scale) : resize_pil_taps(H, outH);
  const int Kh = matlab ? Kv : resize_pil_taps(W, outW);
  // the scratch was sized with resize_matlab_taps_bound of (H, outH) and (W, outW); tables of K taps fit in it when K is within both
  if (matlab && (Kv > resize_matlab_taps_bound(H, outH) || Kv > resize_matlab_taps_bound(W, outW))) {
    set_error("hitsir_resize_f32_matlab: scale %g is too small for a %d x %d image", scale, H, W);
    return 1;
  }
  const size_t smem = matlab ? resize_smem_bytes<float, 1>(Kv, Kh)
                             : (C == 3 ? resize_smem_bytes<uint8_t, 3>(Kv, Kh) : resize_smem_bytes<uint8_t, 1>(Kv, Kh));
  if (smem > (size_t)kMaxSmem) {
    set_error("hitsir_resize: %d x %d -> %d x %d needs %d and %d taps per output, more than a CTA's shared memory holds", H, W, outH, outW,
              Kv, Kh);
    return 1;
  }
  return 0;
}

long long resize_scratch_bytes(int matlab, int H, int W, int outH, int outW) {
  const int Kv = matlab ? resize_matlab_taps_bound(H, outH) : resize_pil_taps(H, outH);
  const int Kh = matlab ? resize_matlab_taps_bound(W, outW) : resize_pil_taps(W, outW);
  return (long long)(table_bytes(outH, Kv) + table_bytes(outW, Kh));
}

int launch_resize_pil(const uint8_t* src, uint8_t* dst, int B, int H, int W, int C, int outH, int outW, void* scratch, cudaStream_t st) {
  AxisSpec sv, sh;
  unsigned char* base = static_cast<unsigned char*>(scratch);
  const int Kv = resize_pil_taps(H, outH), Kh = resize_pil_taps(W, outW);
  const Table tv = make_table(base, outH, Kv, &sv, H, 0.0);
  const Table th = make_table(base + table_bytes(outH, Kv), outW, Kh, &sh, W, 0.0);
  if (launch_taps<true>(sv, sh, st)) return 1;
  return C == 3 ? launch_resample<uint8_t, 3>(src, dst, B, H, W, outH, outW, tv, th, st)
                : launch_resample<uint8_t, 1>(src, dst, B, H, W, outH, outW, tv, th, st);
}

int launch_resize_matlab(const float* src, float* dst, int B, int C, int H, int W, double scale, int outH, int outW, void* scratch,
                         cudaStream_t st) {
  AxisSpec sv, sh;
  unsigned char* base = static_cast<unsigned char*>(scratch);
  const int K = resize_matlab_taps(scale);
  const Table tv = make_table(base, outH, K, &sv, H, scale);
  const Table th = make_table(base + table_bytes(outH, K), outW, K, &sh, W, scale);
  if (launch_taps<false>(sv, sh, st)) return 1;
  return launch_resample<float, 1>(src, dst, B * C, H, W, outH, outW, tv, th, st);
}

}  // namespace hitsir
