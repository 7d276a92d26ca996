// Dense-contraction front end of the tcgen05 kernels (umma_gemm.cu, umma_gemm_tma.cu, conv3_c64.cu): problem description + the
// fused epilogue of the direct-store kernel.
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
enum ActMode : int { ACT_NONE = 0, ACT_GELU = 1, ACT_LRELU = 2 };

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
  // operand views for debugging (no kernel reads them: the kernels take tensor maps)
  const bf16* A; int lda;         // linear: [M, lda]; conv: NHWC base with lda = Cin_pad
  const bf16* Wp; int ldw;        // [n_tiles*BN, ldw]
};

// Row bookkeeping of the direct-store kernel
struct RowInfo {
  bool valid;
  long long grow;   // linear row / NHWC pixel index
  int b, y, x;      // conv coordinates (pixel)
};

__device__ __forceinline__ RowInfo row_info(const GemmParams& p, int m_tile, int r) {
  RowInfo ri;
  if (!p.conv) {
    long long g = (long long)m_tile * 128 + r;
    ri.valid = g < p.M;
    ri.grow = g;
    ri.b = ri.y = ri.x = 0;
  } else {
    int tx = m_tile % p.tiles_x;
    int t2 = m_tile / p.tiles_x;
    int ty = t2 % p.tiles_y;
    int b = t2 / p.tiles_y;
    int y = ty * 8 + (r >> 4), x = tx * 16 + (r & 15);
    ri.valid = (y < p.H) && (x < p.W);
    ri.b = b; ri.y = y; ri.x = x;
    ri.grow = ((long long)b * p.H + y) * p.W + x;
  }
  return ri;
}

// ---------------------------------------------------------------------------
// Fused epilogue for ONE output row (one thread).  `Acc::load16(col0, v)` returns the 16 raw
// accumulators of columns [col0, col0+16) of this row for the current N tile.
// All threads of a warp must call it together (TMEM loads are warp-collective), invalid rows
// simply skip their global stores.
// ---------------------------------------------------------------------------
template <int BN, class Acc>
__device__ __forceinline__ void epilogue_row(const GemmParams& p, Acc& acc, const RowInfo& ri, int n_tile) {
  const int n0 = n_tile * BN;
  if (p.epi == EPI_STORE) {
#pragma unroll 1
    for (int c0 = 0; c0 < BN; c0 += 16) {
      float v[16];
      acc.load16(c0, v);
      if (!ri.valid) continue;
      const int gc = n0 + c0;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        float t = v[i] + __ldg(p.bias + gc + i);
        if (p.act == ACT_GELU) t = gelu_erf(t);
        else if (p.act == ACT_LRELU) t = lrelu(t, p.slope);
        v[i] = t;
      }
      if (p.res != nullptr) {
        const float* rr = p.res + ri.grow * p.ldr + gc;
#pragma unroll
        for (int i = 0; i < 16; ++i)
          if (gc + i < p.n_real) v[i] += __ldg(rr + i);
      }
      if (p.out_f32 != nullptr) {
        float* o = p.out_f32 + ri.grow * p.ldf + gc;
        if (gc + 16 <= p.n_real && (p.ldf & 3) == 0) {
#pragma unroll
          for (int i = 0; i < 16; i += 4) *reinterpret_cast<float4*>(o + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
        } else {
#pragma unroll
          for (int i = 0; i < 16; ++i)
            if (gc + i < p.n_real) o[i] = v[i];
        }
      }
      if (p.out_bf16 != nullptr && gc < p.ldb) {
        uint32_t w[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          float a = (gc + 2 * i < p.n_real) ? v[2 * i] : 0.f;
          float b = (gc + 2 * i + 1 < p.n_real) ? v[2 * i + 1] : 0.f;
          w[i] = pack_bf16x2(a, b);
        }
        uint4* o = reinterpret_cast<uint4*>(p.out_bf16 + ri.grow * p.ldb + gc);
        o[0] = make_uint4(w[0], w[1], w[2], w[3]);
        o[1] = make_uint4(w[4], w[5], w[6], w[7]);
      }
    }
  } else if (p.epi == EPI_MSGATE) {
    // N tile `n_tile` (BN == 160) holds, for the 32 embedding channels c = 32*n_tile + i:
    //   cols [32k, 32k+32), k=0..3 : conv3/5/7/9 outputs, cols [128,160): conv_x (1x1) output.
    // g_k = x_k * sigmoid(x_1 * x_k) + x_k  (hit_sir_pro.py:83-92) -> out_bf16[row, 128*n_tile + 32*k + i]
    // (the [tile][slot][channel] order the packed conv_first.conv_last expects, pack.cu pack_mslast_kernel).
    float x1[32];
    {
      float v[16];
#pragma unroll
      for (int c0 = 128; c0 < 160; c0 += 16) {
        acc.load16(c0, v);
#pragma unroll
        for (int i = 0; i < 16; ++i) x1[c0 + i - 128] = v[i] + __ldg(p.bias + n0 + c0 + i);
      }
    }
#pragma unroll
    for (int c0 = 0; c0 < 128; c0 += 16) {
      float v[16];
      acc.load16(c0, v);
      if (ri.valid) {
        uint32_t w[8];
#pragma unroll
        for (int i = 0; i < 16; i += 2) {
          const float xa = v[i] + __ldg(p.bias + n0 + c0 + i), xb = v[i + 1] + __ldg(p.bias + n0 + c0 + i + 1);
          const float ga = xa * sigmoidf_(x1[(c0 + i) & 31] * xa) + xa, gb = xb * sigmoidf_(x1[(c0 + i + 1) & 31] * xb) + xb;
          w[i >> 1] = pack_bf16x2(ga, gb);
        }
        uint4* o = reinterpret_cast<uint4*>(p.out_bf16 + ri.grow * p.ldb + 128 * n_tile + c0);
        o[0] = make_uint4(w[0], w[1], w[2], w[3]);
        o[1] = make_uint4(w[4], w[5], w[6], w[7]);
      }
    }
  } else {
    // pixel-shuffle epilogues: column co = c*ps*ps + i*ps + j  -> pixel (ps*y+i, ps*x+j), channel c
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
        float t = v[i] + __ldg(p.bias + co);
        if (p.epi == EPI_SHUFFLE_NCHW) {
          const long long oi = (((long long)ri.b * p.shuf_c + c) * oh + oy) * ow + ox;
          p.out_f32[oi] = t * p.out_scale + (p.res_img != nullptr ? __ldg(p.res_img + oi) : p.mean[c & 3]);
        } else {
          if (p.act == ACT_LRELU) t = lrelu(t, p.slope);
          p.out_bf16[(((long long)ri.b * oh + oy) * ow + ox) * p.ldb + c] = __float2bfloat16(t);
        }
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
