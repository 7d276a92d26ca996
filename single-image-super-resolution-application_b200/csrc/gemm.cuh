// Dense-contraction front end of the tcgen05 kernels (umma_gemm.cu, umma_gemm_tma.cu, conv3_c64.cu): problem description + the
// pixel-shuffle epilogue of the direct-store kernel.  Each epilogue kind has one GEMM kernel: EPI_STORE and EPI_MSGATE run on the
// TMA-staged kernel (umma_gemm_tma.cu), the pixel-shuffle heads EPI_SHUFFLE_* on the direct-store kernel (umma_gemm.cu).
//
// One "problem" is  D[M, N] = A[M, K] * Wp[N, K]^T  with bf16 operands and fp32 accumulation:
//   * linear:  A is a token-major activation [M, K] (K padded to a multiple of 64);
//   * conv3x3: implicit GEMM over an NHWC activation [B, H, W, Cin_pad]; K = 9 * Cin_pad
//              (tap-major, k = (ky*3+kx)*Cin_pad + c), zero padding comes from TMA OOB fill.
// Output rows are 128-row tiles: 128 consecutive tokens (linear) or an 8x16 pixel patch (conv).
#pragma once
#include "common.cuh"

namespace hitsir {

enum EpiMode : int {
  EPI_STORE = 0,    // v = act(acc + bias) (+ res)            -> out_f32 / out_bf16
  EPI_MSGATE = 2,   // MultipleSizeConvExtract gate (hit_sir_pro.py:83-92), see epilogue
  EPI_SHUFFLE_NCHW = 3,  // pixel-shuffle(ps) + de-normalise -> NCHW fp32 image
  EPI_SHUFFLE_BF16 = 4,  // pixel-shuffle(ps) -> NHWC bf16 feature map with `shuf_c` channels
};
enum ActMode : int { ACT_NONE = 0, ACT_LRELU = 2 };

struct GemmParams {
  // problem
  int conv;          // 0 linear, 1 conv3x3
  int M;             // linear: number of rows
  int B, H, W;       // conv: NHWC geometry
  int tiles_x, tiles_y;
  int m_tiles, n_tiles;
  int num_kb;        // K / 64
  int b_resident;    // linear, K <= 192, grid % n_tiles == 0: the CTA's weight tile is loaded once and stays in shared memory (umma_gemm_tma.cu)
  int cblocks;       // conv: Cin_pad / 64
  int a_y_off;       // conv: rows of valid halo ABOVE image row 0 in the A tensor map (band mode: the map covers [-a_y_off, H + a_y_off))
  // epilogue
  int epi, act;
  int n_real;        // number of meaningful output columns (of n_tiles*BN)
  float slope;       // leaky-relu slope
  const float* bias; // [n_tiles*BN], zero padded
  const float* res; int ldr;      // fp32 residual rows
  float* out_f32; int ldf;
  bf16* out_bf16; int ldb;        // columns [0, ldb) are written (zeros beyond n_real)
  // shuffle epilogues
  int ps;            // pixel-shuffle factor (1 = none)
  int shuf_c;        // channels after shuffle (NCHW: image channels; BF16: feature channels = ldb)
  float out_scale;   // 1 / img_range
  float mean[4];     // per-channel mean added after scaling (NCHW)
  const float* res_img;   // EPI_SHUFFLE_NCHW, ps == 1: NCHW fp32 image added INSTEAD of the mean (upsampler=None: x + conv_last(res), :1340-1342)
};

// Conv M tiles: 8 x 16 pixels = 128 GEMM rows, row r <-> pixel (y0 + r / 16, x0 + r % 16); tile t runs x fastest, then y, then the
// image.  conv_last_fold (conv3_c64.cu) walks its own tile shape with the same order.
constexpr int kConvTileH = 8, kConvTileW = 16;
struct ConvTile { int b, y0, x0; };
__host__ __device__ __forceinline__ ConvTile conv_tile(int t, int tiles_x, int tiles_y, int th = kConvTileH, int tw = kConvTileW) {
  const int tx = t % tiles_x, t2 = t / tiles_x;
  ConvTile c;
  c.x0 = tx * tw; c.y0 = (t2 % tiles_y) * th; c.b = t2 / tiles_y;
  return c;
}

// Row bookkeeping of the direct-store kernel
struct RowInfo {
  bool valid;
  int b, y, x;      // conv coordinates (pixel)
};

__device__ __forceinline__ RowInfo row_info(const GemmParams& p, int m_tile, int r) {
  RowInfo ri;
  if (!p.conv) {
    ri.valid = (long long)m_tile * 128 + r < p.M;
    ri.b = ri.y = ri.x = 0;
  } else {
    const ConvTile t = conv_tile(m_tile, p.tiles_x, p.tiles_y);
    const int b = t.b, y = t.y0 + (r >> 4), x = t.x0 + (r & 15);
    ri.valid = (y < p.H) && (x < p.W);
    ri.b = b; ri.y = y; ri.x = x;
  }
  return ri;
}

// ---------------------------------------------------------------------------
// Pixel-shuffle epilogue for ONE output row (one thread).  `Acc::load16(col0, v)` returns the 16 raw
// accumulators of columns [col0, col0+16) of this row for the current N tile.
// All threads of a warp must call it together (TMEM loads are warp-collective), invalid rows
// simply skip their global stores.
// ---------------------------------------------------------------------------
template <int BN, class Acc>
__device__ __forceinline__ void epilogue_row(const GemmParams& p, Acc& acc, const RowInfo& ri, int n_tile) {
  const int n0 = n_tile * BN;
  // column co = c*ps*ps + i*ps + j  -> pixel (ps*y+i, ps*x+j), channel c
  const int ps = p.ps, pss = ps * ps;
  const int oh = p.H * ps, ow = p.W * ps;
#pragma unroll 1
  for (int c0 = 0; c0 < BN; c0 += 16) {
    float v[16];
    acc.load16(c0, v);
    if (!ri.valid) continue;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const int co = n0 + c0 + i;
      if (co >= p.n_real) continue;
      const int c = co / pss, rem = co - c * pss;
      const int oy = ri.y * ps + rem / ps, ox = ri.x * ps + rem % ps;
      const float t = v[i] + __ldg(p.bias + co);
      if (p.epi == EPI_SHUFFLE_NCHW) {
        const long long oi = (((long long)ri.b * p.shuf_c + c) * oh + oy) * ow + ox;
        p.out_f32[oi] = t * p.out_scale + (p.res_img != nullptr ? __ldg(p.res_img + oi) : p.mean[c & 3]);
      } else {
        p.out_bf16[(((long long)ri.b * oh + oy) * ow + ox) * p.ldb + c] = __float2bfloat16(t);
      }
    }
  }
}

// host-side launchers (umma_gemm.cu)
struct TensorMaps {
  CUtensorMap a, b;
};
int make_tmap_2d(CUtensorMap* m, const void* base, uint64_t inner, uint64_t outer, uint64_t pitch_bytes, uint32_t box_inner, uint32_t box_outer);
int make_tmap_nhwc(CUtensorMap* m, const void* base, int B, int H, int W, int Cpad, uint32_t box_c, uint32_t box_w, uint32_t box_h);
int make_tmap_2d_t(CUtensorMap* m, const void* base, int elem_bytes, uint64_t inner, uint64_t outer, uint64_t pitch_bytes, uint32_t box_inner, uint32_t box_outer);
int make_tmap_nhwc_t(CUtensorMap* m, const void* base, int elem_bytes, int B, int H, int W, int C, int ldc, uint32_t box_c, uint32_t box_w, uint32_t box_h);
// bf16 NHWC view with explicit pixel / row / image strides (bytes): the four phase sub-lattices of a x2 upsampled map
int make_tmap_nhwc_strided(CUtensorMap* m, const void* base, int B, int H, int W, int C, uint64_t pix_bytes, uint64_t row_bytes, uint64_t img_bytes,
                           uint32_t box_c, uint32_t box_w, uint32_t box_h);
// x2 nearest upsampling + 3x3 conv 64 -> 64 + bias + LeakyReLU as four 2x2 phase convs on the LR map (conv3_c64.cu); A [B,H,W,64], out [B,2H,2W,64]
int launch_conv3_c64_up(const GemmParams& p, const bf16* A, const CUtensorMap& tb, int num_sms, cudaStream_t st);
// conv_last 64 -> n_real <= 4 with the nine taps folded into N (conv3_c64.cu); tb = folded filters [48][64], out_f32 NCHW (EPI_SHUFFLE_NCHW, ps = 1)
int launch_conv_last_fold(const GemmParams& p, const bf16* A, const CUtensorMap& tb, int num_sms, cudaStream_t st);
int launch_conv3_c64(int BN, const GemmParams& p, const bf16* A, const CUtensorMap& tb, int num_sms, cudaStream_t st);
int launch_umma_gemm_tma(int BN, const GemmParams& p, const CUtensorMap* maps, int num_sms, cudaStream_t st);
// proj + norm1 + residual and fc1 + GELU of one transformer block (proj_fc1.cu); maps: {outsc [M,192] bf16 box {64,128}, Wp and W1 packed
// (box {64,192}), residual x and stream x' fp32 [M,180] box {32,128}, h1 bf16 [M,384] box {64,128}}
struct ProjFc1Params {
  int m_tiles;
  const float* bias_p;               // [192], zero padded
  const float* gamma; const float* beta;   // norm1, [180]
  const float* bias1;                // [384], zero padded
};
int launch_proj_fc1(const ProjFc1Params& p, const CUtensorMap* maps, int num_sms, cudaStream_t st);
int launch_umma_gemm(int BN, const GemmParams& p, const CUtensorMap& ta, const CUtensorMap& tb, int num_sms, cudaStream_t st);

}  // namespace hitsir
