// 3x3 convolution over a 64-channel NHWC bf16 map (the HR stage of the 'nearest+conv' / 'pixelshuffle' upsamplers:
// conv_up1, conv_up2, conv_hr 64 -> 64 with LeakyReLU, conv_last 64 -> in_chans; /root/reference/models/hit_sir_pro.py:1326-1334)
// as an implicit GEMM on tcgen05, specialised for Cin = 64:
//   * the whole filter bank (9 taps x BN x 64 bf16 = 72 KB for BN = 64) stays resident in shared memory for the life of the
//     persistent CTA -- the generic kernel re-fetched 8 KB of weights per tap per tile from L2;
//   * one TMA box per horizontal tap offset kx covers all three vertical taps: a (8+2) x 16 pixel box, whose rows ky*16 ..
//     ky*16+127 are the A operand of tap (ky, kx) (descriptor start + ky * 2 KB, still 1024-byte aligned).  Every input pixel
//     is therefore fetched 3.75x per tile instead of 9x; the generic kernel was bound by L2->SM traffic (~10 TB/s), not by HBM.
// Out-of-image taps are TMA out-of-bounds zero fill (= the conv's zero padding).
// bias + LeakyReLU -> bf16 NHWC via a swizzled box and TMA store.  (conv_last, 64 -> in_chans, has its own kernel below: with N = 16
// this one spent 36 tensor-core instructions of ~53 cycles on 128 pixels.)
#include "gemm.cuh"

namespace hitsir {

namespace {

constexpr int kATile = 160 * 128;          // (8 + 2) rows x 16 pixels x 64 ch bf16
constexpr int kAStages = 4;                // deeper rings (5, 9) measured no faster: the kernel is bound by the tcgen05 pipe (72 % busy), not by the ring
constexpr int kBoxBytes = 128 * 128;
constexpr int kNBox = 3;

template <int BN>
struct Cfg {
  static constexpr int kBBytes = 9 * BN * 128;                      // resident filter bank
  static constexpr int kOffA = (kBBytes + 1023) / 1024 * 1024;
  static constexpr int kOffBox = kOffA + kAStages * kATile;
  static constexpr int kOffBias = kOffBox + kNBox * kBoxBytes;
  static constexpr int kOffBars = kOffBias + 64 * 4;
  static constexpr int kSmemBytes = kOffBars + 32 * 8 + 16 + 1024;
  static_assert(2 * kAStages + 4 + 2 * kNBox + 1 <= 32, "barrier slots");
  static_assert(kSmemBytes <= 232448, "smem budget");
  static constexpr int kTmemCols = 128;
};

template <int BN>
__global__ void __launch_bounds__(384, 1)
conv3_c64_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b, const __grid_constant__ CUtensorMap tmap_o,
                 const GemmParams p) {
  using C = Cfg<BN>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sb = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sp = smem_raw + (sb - smem_u32(smem_raw));
  float* s_bias = reinterpret_cast<float*>(sp + C::kOffBias);
  const uint32_t bar0 = sb + C::kOffBars;
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (kAStages + s); };
  auto tfull_bar = [&](int s) { return bar0 + 8u * (2 * kAStages + s); };
  auto tempty_bar = [&](int s) { return bar0 + 8u * (2 * kAStages + 2 + s); };
  auto box_free = [&](int s) { return bar0 + 8u * (2 * kAStages + 4 + s); };
  auto box_ready = [&](int s) { return bar0 + 8u * (2 * kAStages + 4 + kNBox + s); };
  const uint32_t b_full = bar0 + 8u * (2 * kAStages + 4 + 2 * kNBox);
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(sp + C::kOffBars + 32 * 8);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int total = p.m_tiles;
  if (warp == 0 && lane == 0) { tma_prefetch_desc(&tmap_a); tma_prefetch_desc(&tmap_b); tma_prefetch_desc(&tmap_o); }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < kAStages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(tfull_bar(s), 1); mbar_init(tempty_bar(s), 8); }
    for (int s = 0; s < kNBox; ++s) { mbar_init(box_free(s), 1); mbar_init(box_ready(s), 8); }
    mbar_init(b_full, 1);
    fence_barrier_init();
  }
  if (warp == 2) { tmem_alloc(smem_u32(tmem_ptr_smem), C::kTmemCols); tmem_relinquish(); }
  for (int i = threadIdx.x; i < 64; i += blockDim.x) s_bias[i] = i < BN ? p.bias[i] : 0.f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    if (lane == 0) {
      // ===================== producer: filter bank once, then one halo box per (tile, kx) =====================
      mbar_expect_tx(b_full, (uint32_t)C::kBBytes);
      for (int tap = 0; tap < 9; ++tap) tma_load_2d(sb + tap * BN * 128, &tmap_b, b_full, tap * 64, 0);
      uint32_t cnt = 0;
      for (int t = blockIdx.x; t < total; t += gridDim.x) {
        const auto [b, y0, x0] = conv_tile(t, p.tiles_x, p.tiles_y);
        for (int kx = 0; kx < 3; ++kx, ++cnt) {
          const int s = (int)(cnt % kAStages);
          mbar_wait(empty_bar(s), ((cnt / kAStages) & 1u) ^ 1u);
          mbar_expect_tx(full_bar(s), kATile);
          tma_load_4d(sb + C::kOffA + s * kATile, &tmap_a, full_bar(s), 0, x0 + kx - 1, y0 - 1 + p.a_y_off, b);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ===================== MMA issuer: 3 (kx) x 3 (ky) x 4 (k-steps) per tile =====================
      constexpr uint32_t idesc = umma_idesc_bf16(128, BN);
      mbar_wait(b_full, 0u);
      uint32_t cnt = 0;
      int it = 0;
      for (int t = blockIdx.x; t < total; t += gridDim.x, ++it) {
        const int as = it & 1;
        mbar_wait(tempty_bar(as), (((uint32_t)(it >> 1)) & 1u) ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(as * BN);
        for (int kx = 0; kx < 3; ++kx, ++cnt) {
          const int s = (int)(cnt % kAStages);
          mbar_wait(full_bar(s), (cnt / kAStages) & 1u);
          tc_fence_after();
          const uint32_t sa = sb + C::kOffA + s * kATile;
#pragma unroll
          for (int ky = 0; ky < 3; ++ky) {
            const uint64_t adesc = umma_desc_sw128(sa + ky * 2048);
            const uint64_t bdesc = umma_desc_sw128(sb + (ky * 3 + kx) * BN * 128);
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_bf16(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (kx | ky | k) != 0 ? 1u : 0u);
          }
          umma_commit(empty_bar(s));
        }
        umma_commit(tfull_bar(as));
      }
    }
  } else if (warp == 3) {
    if (lane == 0) {
      // ===================== TMA store of finished boxes =====================
      uint32_t u = 0;
      for (int t = blockIdx.x; t < total; t += gridDim.x, ++u) {
        const auto [b, y0, x0] = conv_tile(t, p.tiles_x, p.tiles_y);
        const int s = (int)(u % kNBox);
        mbar_wait(box_ready(s), (u / kNBox) & 1u);
        tma_store_4d(&tmap_o, sb + C::kOffBox + s * kBoxBytes, 0, x0, y0, b);
        tma_commit();
        tma_wait_read<1>();                                // groups retire in order: the previous box is free again
        if (u >= 1) mbar_arrive(box_free((int)((u - 1) % kNBox)));
      }
      tma_wait_all0();
    }
  } else if (warp >= 4) {
    // ===================== epilogue: 8 warps, two per TMEM lane quarter =====================
    const int q = warp & 3, hs = (warp - 4) >> 2;
    const int r = q * 32 + lane;
    int it = 0;
    uint32_t u = 0;
    for (int t = blockIdx.x; t < total; t += gridDim.x, ++it, ++u) {
      const int as = it & 1;
      mbar_wait(tfull_bar(as), ((uint32_t)(it >> 1)) & 1u);
      tc_fence_after();
      const uint32_t tacc = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * BN);
      float v[32];
      tmem_ld32(tacc + 32 * hs, v);
      tc_fence_before();
      mbar_arrive_warp(tempty_bar(as));
#pragma unroll
      for (int i = 0; i < 32; ++i) { const float x = v[i] + s_bias[32 * hs + i]; v[i] = p.act == ACT_LRELU ? lrelu(x, p.slope) : x; }
      const int s = (int)(u % kNBox);
      if (u >= (uint32_t)kNBox) mbar_wait(box_free(s), ((u / kNBox) - 1u) & 1u);
      uint8_t* row = sp + C::kOffBox + s * kBoxBytes + r * 128;
#pragma unroll
      for (int ch = 0; ch < 4; ++ch) {
        const uint4 o = make_uint4(pack_bf16x2(v[8 * ch], v[8 * ch + 1]), pack_bf16x2(v[8 * ch + 2], v[8 * ch + 3]),
                                   pack_bf16x2(v[8 * ch + 4], v[8 * ch + 5]), pack_bf16x2(v[8 * ch + 6], v[8 * ch + 7]));
        *reinterpret_cast<uint4*>(row + (((uint32_t)(4 * hs + ch) ^ (uint32_t)(r & 7)) << 4)) = o;
      }
      fence_proxy_async_smem();
      mbar_arrive_warp(box_ready(s));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, C::kTmemCols);
  }
}

// ---------------------------------------------------------------------------------------------------------------------------
// x2 nearest upsampling + 3x3 conv 64 -> 64 + bias + LeakyReLU without the upsampled map (conv_up1 / conv_up2, :1331-1332).
// Output phase (a, b) = (Y & 1, X & 1) of the HR map is a 2x2 conv of the LR map with the phase filters of pack_subpixel_kernel:
// 16 instead of 36 tap-MMAs per HR pixel quad, the LR map is read instead of a 4x larger replicated one, and the upsample2 pass
// (write + read of the replicated map) is gone.  Per 8 x 16 LR tile the three kx boxes of the plain kernel feed four accumulators
// [128 x 64] (one per phase, 256 TMEM columns, double-buffered = all 512); box kx serves the phases with dx = kx - 1 in {b - 1, b}.
// The four results leave through four tensor maps over the HR map (pixel stride 2, row stride 2, base offset (a, b)), so the TMA
// store does the interleaving and clips at the LR image size.
constexpr int kUpAStages = 3;
constexpr int kUpNBox = 2;
struct UpCfg {
  static constexpr int kBBytes = 16 * 64 * 128;                       // resident phase filters: 4 phases x 4 taps x [64 x 64]
  static constexpr int kOffA = kBBytes;
  static constexpr int kOffBox = kOffA + kUpAStages * kATile;
  static constexpr int kOffBias = kOffBox + kUpNBox * kBoxBytes;
  static constexpr int kOffBars = kOffBias + 64 * 4;
  static constexpr int kSmemBytes = kOffBars + 32 * 8 + 16 + 1024;
};
static_assert(UpCfg::kSmemBytes <= 232448 && UpCfg::kOffA % 1024 == 0 && UpCfg::kOffBox % 1024 == 0, "smem budget / alignment");

__global__ void __launch_bounds__(384, 1)
conv3_c64_up_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b, const __grid_constant__ CUtensorMap tmap_o0,
                    const __grid_constant__ CUtensorMap tmap_o1, const __grid_constant__ CUtensorMap tmap_o2, const __grid_constant__ CUtensorMap tmap_o3,
                    const GemmParams p) {
  using C = UpCfg;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sb = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sp = smem_raw + (sb - smem_u32(smem_raw));
  float* s_bias = reinterpret_cast<float*>(sp + C::kOffBias);
  const uint32_t bar0 = sb + C::kOffBars;
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (kUpAStages + s); };
  auto tfull_bar = [&](int s) { return bar0 + 8u * (2 * kUpAStages + s); };
  auto tempty_bar = [&](int s) { return bar0 + 8u * (2 * kUpAStages + 2 + s); };
  auto box_free = [&](int s) { return bar0 + 8u * (2 * kUpAStages + 4 + s); };
  auto box_ready = [&](int s) { return bar0 + 8u * (2 * kUpAStages + 4 + kUpNBox + s); };
  const uint32_t b_full = bar0 + 8u * (2 * kUpAStages + 4 + 2 * kUpNBox);
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(sp + C::kOffBars + 32 * 8);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int total = p.m_tiles;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a); tma_prefetch_desc(&tmap_b);
    tma_prefetch_desc(&tmap_o0); tma_prefetch_desc(&tmap_o1); tma_prefetch_desc(&tmap_o2); tma_prefetch_desc(&tmap_o3);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < kUpAStages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(tfull_bar(s), 1); mbar_init(tempty_bar(s), 8); }
    for (int s = 0; s < kUpNBox; ++s) { mbar_init(box_free(s), 1); mbar_init(box_ready(s), 8); }
    mbar_init(b_full, 1);
    fence_barrier_init();
  }
  if (warp == 2) { tmem_alloc(smem_u32(tmem_ptr_smem), 512); tmem_relinquish(); }
  for (int i = threadIdx.x; i < 64; i += blockDim.x) s_bias[i] = p.bias[i];
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    if (lane == 0) {
      // ===================== producer: phase filters once, then one LR halo box per (tile, kx) =====================
      mbar_expect_tx(b_full, (uint32_t)C::kBBytes);
      for (int tap = 0; tap < 16; ++tap) tma_load_2d(sb + tap * 64 * 128, &tmap_b, b_full, tap * 64, 0);
      uint32_t cnt = 0;
      for (int t = blockIdx.x; t < total; t += gridDim.x) {
        const auto [b, y0, x0] = conv_tile(t, p.tiles_x, p.tiles_y);
        for (int kx = 0; kx < 3; ++kx, ++cnt) {
          const int s = (int)(cnt % kUpAStages);
          mbar_wait(empty_bar(s), ((cnt / kUpAStages) & 1u) ^ 1u);
          mbar_expect_tx(full_bar(s), kATile);
          tma_load_4d(sb + C::kOffA + s * kATile, &tmap_a, full_bar(s), 0, x0 + kx - 1, y0 - 1 + p.a_y_off, b);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ===================== MMA issuer: LR offset (dy, dx) = (ky - 1, kx - 1) feeds phase (a, b) iff ky - a, kx - b in {0, 1} =====================
      constexpr uint32_t idesc = umma_idesc_bf16(128, 64);
      mbar_wait(b_full, 0u);
      uint32_t cnt = 0;
      int it = 0;
      for (int t = blockIdx.x; t < total; t += gridDim.x, ++it) {
        const int as = it & 1;
        mbar_wait(tempty_bar(as), (((uint32_t)(it >> 1)) & 1u) ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(as * 256);
#pragma unroll
        for (int kx = 0; kx < 3; ++kx, ++cnt) {
          const int s = (int)(cnt % kUpAStages);
          mbar_wait(full_bar(s), (cnt / kUpAStages) & 1u);
          tc_fence_after();
          const uint32_t sa = sb + C::kOffA + s * kATile;
#pragma unroll
          for (int ky = 0; ky < 3; ++ky) {
            const uint64_t adesc = umma_desc_sw128(sa + ky * 2048);
#pragma unroll
            for (int a = 0; a < 2; ++a) {
              const int dyi = ky - a;
              if (dyi < 0 || dyi > 1) continue;
#pragma unroll
              for (int b = 0; b < 2; ++b) {
                const int dxi = kx - b;
                if (dxi < 0 || dxi > 1) continue;
                const int ph = 2 * a + b;
                const uint64_t bdesc = umma_desc_sw128(sb + ((ph * 4 + dyi * 2 + dxi) * 64) * 128);
#pragma unroll
                for (int k = 0; k < 4; ++k)      // (dyi, dxi) = (0, 0) is the first tap of every phase in this loop order
                  umma_bf16(d_tmem + (uint32_t)(ph * 64), adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (dyi | dxi | k) != 0 ? 1u : 0u);
              }
            }
          }
          umma_commit(empty_bar(s));
        }
        umma_commit(tfull_bar(as));
      }
    }
  } else if (warp == 3) {
    if (lane == 0) {
      // ===================== TMA store: box u = (tile, phase) through the phase's strided view of the HR map =====================
      uint32_t u = 0;
      for (int t = blockIdx.x; t < total; t += gridDim.x) {
        const auto [b, y0, x0] = conv_tile(t, p.tiles_x, p.tiles_y);
        for (int ph = 0; ph < 4; ++ph, ++u) {
          const int s = (int)(u % kUpNBox);
          mbar_wait(box_ready(s), (u / kUpNBox) & 1u);
          const CUtensorMap* tm = ph == 0 ? &tmap_o0 : ph == 1 ? &tmap_o1 : ph == 2 ? &tmap_o2 : &tmap_o3;
          tma_store_4d(tm, sb + C::kOffBox + s * kBoxBytes, 0, x0, y0, b);
          tma_commit();
          tma_wait_read<1>();                                // groups retire in order: the previous box is free again
          if (u >= 1) mbar_arrive(box_free((int)((u - 1) % kUpNBox)));
        }
      }
      tma_wait_all0();
    }
  } else if (warp >= 4) {
    // ===================== epilogue: 8 warps, two per TMEM lane quarter; four phase boxes per tile =====================
    const int q = warp & 3, hs = (warp - 4) >> 2;
    const int r = q * 32 + lane;
    int it = 0;
    uint32_t u = 0;
    for (int t = blockIdx.x; t < total; t += gridDim.x, ++it) {
      const int as = it & 1;
      mbar_wait(tfull_bar(as), ((uint32_t)(it >> 1)) & 1u);
      tc_fence_after();
      const uint32_t tacc = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * 256);
#pragma unroll 1
      for (int ph = 0; ph < 4; ++ph, ++u) {
        float v[32];
        tmem_ld32(tacc + 64 * ph + 32 * hs, v);
        if (ph == 3) { tc_fence_before(); mbar_arrive_warp(tempty_bar(as)); }
#pragma unroll
        for (int i = 0; i < 32; ++i) { const float x = v[i] + s_bias[32 * hs + i]; v[i] = p.act == ACT_LRELU ? lrelu(x, p.slope) : x; }
        const int s = (int)(u % kUpNBox);
        if (u >= (uint32_t)kUpNBox) mbar_wait(box_free(s), ((u / kUpNBox) - 1u) & 1u);
        uint8_t* row = sp + C::kOffBox + s * kBoxBytes + r * 128;
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {
          const uint4 o = make_uint4(pack_bf16x2(v[8 * ch], v[8 * ch + 1]), pack_bf16x2(v[8 * ch + 2], v[8 * ch + 3]),
                                     pack_bf16x2(v[8 * ch + 4], v[8 * ch + 5]), pack_bf16x2(v[8 * ch + 6], v[8 * ch + 7]));
          *reinterpret_cast<uint4*>(row + (((uint32_t)(4 * hs + ch) ^ (uint32_t)(r & 7)) << 4)) = o;
        }
        fence_proxy_async_smem();
        mbar_arrive_warp(box_ready(s));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ---------------------------------------------------------------------------------------------------------------------------
// conv_last (64 -> in_chans <= 4, :1334 / :1241) with the nine taps folded into the N dimension.  The plain kernel issues 36 MMAs of
// N = 16 per 128 output pixels, and a tcgen05.mma with shared-memory A costs ~53 cycles however small N is (ncu: tensor-core pipe busy
// 73 %, math 12 %, profiles/r2_ncu_full_hr_convs_summary.csv).  Here every INPUT pixel q of an (6+2) x (30+2) halo tile is multiplied
// once by all taps, P[q][tap][co] = a_q . w[co][:][tap] (one [256 x 64] x [64 x 48] contraction = 8 MMAs), and the epilogue adds the nine
// shifted partial products per output pixel from shared memory: out[y][x][co] = b[co] + sum_t P[(y+ky, x+kx)][t][co].  8 instead of
// 50 MMAs per 180 outputs, and one 32 KB halo box per tile instead of three 20 KB ones (1.4x instead of 3.75x re-fetch).
constexpr int kFoldTW = 30, kFoldTH = 6;                // output tile; halo box 32 x 8 pixels = 256 rows = two M blocks
constexpr int kFoldA = 256 * 128;
constexpr int kFoldStages = 4;
constexpr int kFoldN = 48;                              // 9 taps x 4 output channels, padded to a multiple of 16
constexpr int kFoldPRow = 36;                           // floats per halo pixel in the partial-product buffer (144 B: float4 accesses of a quarter warp hit 32 banks)
struct FoldCfg {
  static constexpr int kBBytes = kFoldN * 128;
  static constexpr int kOffA = kBBytes;                                       // 6144: 1024-byte aligned
  static constexpr int kOffP = kOffA + kFoldStages * kFoldA;
  static constexpr int kOffBars = kOffP + 2 * 256 * kFoldPRow * 4;
  static constexpr int kSmemBytes = kOffBars + 16 * 8 + 16 + 1024;
};
static_assert(FoldCfg::kSmemBytes <= 232448 && FoldCfg::kOffA % 1024 == 0, "smem budget / alignment");

__global__ void __launch_bounds__(384, 1)
conv_last_fold_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b, const GemmParams p) {
  using C = FoldCfg;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sb = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sp = smem_raw + (sb - smem_u32(smem_raw));
  const uint32_t bar0 = sb + C::kOffBars;
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (kFoldStages + s); };
  auto tfull_bar = [&](int s) { return bar0 + 8u * (2 * kFoldStages + s); };
  auto tempty_bar = [&](int s) { return bar0 + 8u * (2 * kFoldStages + 2 + s); };
  const uint32_t b_full = bar0 + 8u * (2 * kFoldStages + 4);
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(sp + C::kOffBars + 16 * 8);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int total = p.m_tiles;
  if (warp == 0 && lane == 0) { tma_prefetch_desc(&tmap_a); tma_prefetch_desc(&tmap_b); }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < kFoldStages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(tfull_bar(s), 1); mbar_init(tempty_bar(s), 8); }
    mbar_init(b_full, 1);
    fence_barrier_init();
  }
  if (warp == 2) { tmem_alloc(smem_u32(tmem_ptr_smem), 256); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    if (lane == 0) {
      // ===================== producer: folded filters once, then one halo box per tile =====================
      mbar_expect_tx(b_full, (uint32_t)C::kBBytes);
      tma_load_2d(sb, &tmap_b, b_full, 0, 0);
      uint32_t cnt = 0;
      for (int t = blockIdx.x; t < total; t += gridDim.x, ++cnt) {
        const auto [b, y0, x0] = conv_tile(t, p.tiles_x, p.tiles_y, kFoldTH, kFoldTW);
        const int s = (int)(cnt % kFoldStages);
        mbar_wait(empty_bar(s), ((cnt / kFoldStages) & 1u) ^ 1u);
        mbar_expect_tx(full_bar(s), kFoldA);
        tma_load_4d(sb + C::kOffA + s * kFoldA, &tmap_a, full_bar(s), 0, x0 - 1, y0 - 1 + p.a_y_off, b);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ===================== MMA issuer: P[256 x 48] = A[256 x 64] Wfold^T, two M blocks x four k-steps =====================
      constexpr uint32_t idesc = umma_idesc_bf16(128, kFoldN);
      mbar_wait(b_full, 0u);
      const uint64_t bdesc = umma_desc_sw128(sb);
      uint32_t cnt = 0;
      for (int t = blockIdx.x; t < total; t += gridDim.x, ++cnt) {
        const int as = (int)(cnt & 1u);
        const int s = (int)(cnt % kFoldStages);
        mbar_wait(tempty_bar(as), ((cnt >> 1) & 1u) ^ 1u);
        mbar_wait(full_bar(s), (cnt / kFoldStages) & 1u);
        tc_fence_after();
        const uint32_t sa = sb + C::kOffA + s * kFoldA;
#pragma unroll
        for (int mb = 0; mb < 2; ++mb) {
          const uint64_t adesc = umma_desc_sw128(sa + mb * 16384);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16(tmem_base + (uint32_t)(as * 2 * kFoldN + mb * kFoldN), adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, k != 0 ? 1u : 0u);
        }
        umma_commit(empty_bar(s));
        umma_commit(tfull_bar(as));
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue (8 warps): partial products TMEM -> shared memory, then 9-tap gather per output pixel =====================
    const int q = warp & 3, mb = (warp - 4) >> 2;
    const int row = mb * 128 + q * 32 + lane;                // halo pixel of this thread in step 1
    const int tid = threadIdx.x - 128;                       // output pixel of this thread in step 2 (first 180 threads)
    const int oy = tid / kFoldTW, ox = tid - oy * kFoldTW;
    float bias[4], mean[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) { bias[c] = c < p.n_real ? p.bias[c] : 0.f; mean[c] = p.mean[c]; }
    uint32_t cnt = 0;
    for (int t = blockIdx.x; t < total; t += gridDim.x, ++cnt) {
      const int as = (int)(cnt & 1u);
      float* P = reinterpret_cast<float*>(sp + C::kOffP) + (size_t)as * 256 * kFoldPRow;
      mbar_wait(tfull_bar(as), (cnt >> 1) & 1u);
      tc_fence_after();
      {
        const uint32_t tacc = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * 2 * kFoldN + mb * kFoldN);
        uint32_t r0[16], r1[16], r2[16];
        tmem_ld16_nw(tacc, r0); tmem_ld16_nw(tacc + 16, r1); tmem_ld16_nw(tacc + 32, r2);
        tmem_ld_wait();
        reg_fence16(r0); reg_fence16(r1); reg_fence16(r2);
        tc_fence_before();
        mbar_arrive_warp(tempty_bar(as));
        uint4* dst = reinterpret_cast<uint4*>(P + (size_t)row * kFoldPRow);
#pragma unroll
        for (int i = 0; i < 4; ++i) dst[i] = make_uint4(r0[4 * i], r0[4 * i + 1], r0[4 * i + 2], r0[4 * i + 3]);
#pragma unroll
        for (int i = 0; i < 4; ++i) dst[4 + i] = make_uint4(r1[4 * i], r1[4 * i + 1], r1[4 * i + 2], r1[4 * i + 3]);
        dst[8] = make_uint4(r2[0], r2[1], r2[2], r2[3]);      // columns 32..35 = tap 8; 36..47 are padding
      }
      named_bar_sync(1, 256);                        // the eight epilogue warps only; P is double-buffered by tile parity
      if (tid < kFoldTW * kFoldTH) {
        const auto [b, y0, x0] = conv_tile(t, p.tiles_x, p.tiles_y, kFoldTH, kFoldTW);
        const int y = y0 + oy, x = x0 + ox;
        float4 acc = make_float4(bias[0], bias[1], bias[2], bias[3]);
#pragma unroll
        for (int ky = 0; ky < 3; ++ky)
#pragma unroll
          for (int kx = 0; kx < 3; ++kx) {
            const float4 v = *reinterpret_cast<const float4*>(P + (size_t)((oy + ky) * 32 + ox + kx) * kFoldPRow + (ky * 3 + kx) * 4);
            acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
          }
        if (y < p.H && x < p.W) {
          const float o[4] = {acc.x, acc.y, acc.z, acc.w};
#pragma unroll
          for (int c = 0; c < 4; ++c)
            if (c < p.n_real) p.out_f32[(((long long)b * p.shuf_c + c) * p.H + y) * p.W + x] = o[c] * p.out_scale + mean[c];
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 256);
  }
}

template <int BN>
int launch_bn(const GemmParams& p, const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& to, int num_sms, cudaStream_t st) {
  using C = Cfg<BN>;
  static unsigned long long configured = 0;
  if (ensure_dynamic_smem(conv3_c64_kernel<BN>, C::kSmemBytes, &configured)) return 1;
  const int grid = p.m_tiles < num_sms ? p.m_tiles : num_sms;
  if (grid <= 0) return 0;
  conv3_c64_kernel<BN><<<grid, 384, C::kSmemBytes, st>>>(ta, tb, to, p);
  HITSIR_CHECK(cudaGetLastError());
  return 0;
}

}  // namespace

// A: NHWC bf16 [B,H,W,64]; tb: packed weights [64][576] with a {64, 64} box; out_bf16 [B,H,W,64]
int launch_conv3_c64(int BN, const GemmParams& p, const bf16* A, const CUtensorMap& tb, int num_sms, cudaStream_t st) {
  CUtensorMap ta, to;
  if (BN != 64) { set_error("launch_conv3_c64: unsupported N tile %d", BN); return 1; }
  // band mode: A points at image row 0 of a buffer that has a_y_off valid halo rows above and below (engine.cu conv3)
  if (make_tmap_nhwc(&ta, A - (size_t)p.a_y_off * p.W * 64, p.B, p.H + 2 * p.a_y_off, p.W, 64, 64, 16, 10)) return 1;
  if (make_tmap_nhwc(&to, p.out_bf16, p.B, p.H, p.W, 64, 64, 16, 8)) return 1;
  return launch_bn<64>(p, ta, tb, to, num_sms, st);
}

// A: NHWC bf16 [B,H,W,64] (the LR map; band mode: a_y_off valid halo rows above and below); tb: phase filters [64][1024] with a {64, 64} box;
// out_bf16: [B,2H,2W,64]
int launch_conv3_c64_up(const GemmParams& p, const bf16* A, const CUtensorMap& tb, int num_sms, cudaStream_t st) {
  static unsigned long long configured = 0;
  if (ensure_dynamic_smem(conv3_c64_up_kernel, UpCfg::kSmemBytes, &configured)) return 1;
  CUtensorMap ta, to[4];
  if (make_tmap_nhwc(&ta, A - (size_t)p.a_y_off * p.W * 64, p.B, p.H + 2 * p.a_y_off, p.W, 64, 64, 16, 10)) return 1;
  const uint64_t pix = 2 * 64 * sizeof(bf16), row = (uint64_t)2 * (2 * p.W) * 64 * sizeof(bf16), img = (uint64_t)(2 * p.H) * (2 * p.W) * 64 * sizeof(bf16);
  for (int ph = 0; ph < 4; ++ph)
    if (make_tmap_nhwc_strided(&to[ph], p.out_bf16 + ((size_t)(ph >> 1) * 2 * p.W + (ph & 1)) * 64, p.B, p.H, p.W, 64, pix, row, img, 64, 16, 8)) return 1;
  const int grid = p.m_tiles < num_sms ? p.m_tiles : num_sms;
  if (grid <= 0) return 0;
  conv3_c64_up_kernel<<<grid, 384, UpCfg::kSmemBytes, st>>>(ta, tb, to[0], to[1], to[2], to[3], p);
  HITSIR_CHECK(cudaGetLastError());
  return 0;
}

// conv_last with folded taps: A NHWC bf16 [B,H,W,64]; tb: folded filters [48][64] (row = tap * 4 + co) with a {64, 48} box; out_f32 NCHW image
int launch_conv_last_fold(const GemmParams& p0, const bf16* A, const CUtensorMap& tb, int num_sms, cudaStream_t st) {
  static unsigned long long configured = 0;
  if (ensure_dynamic_smem(conv_last_fold_kernel, FoldCfg::kSmemBytes, &configured)) return 1;
  GemmParams p = p0;
  p.tiles_x = (p.W + kFoldTW - 1) / kFoldTW; p.tiles_y = (p.H + kFoldTH - 1) / kFoldTH;
  const long long total = (long long)p.B * p.tiles_x * p.tiles_y;
  if (total > 2147483647LL) { set_error("launch_conv_last_fold: too many tiles"); return 1; }
  p.m_tiles = (int)total;
  CUtensorMap ta;
  if (make_tmap_nhwc(&ta, A - (size_t)p.a_y_off * p.W * 64, p.B, p.H + 2 * p.a_y_off, p.W, 64, 64, 32, 8)) return 1;
  const int grid = p.m_tiles < num_sms ? p.m_tiles : num_sms;
  if (grid <= 0) return 0;
  conv_last_fold_kernel<<<grid, 384, FoldCfg::kSmemBytes, st>>>(ta, tb, p);
  HITSIR_CHECK(cudaGetLastError());
  return 0;
}

}  // namespace hitsir
