// tcgen05 contraction kernel with a TMA-staged epilogue (EPI_STORE / EPI_MSGATE).
//
// Same mainloop as umma_gemm.cu (TMA -> 128B-swizzled smem -> tcgen05.mma -> TMEM, double-buffered
// accumulators).  The difference is how results leave the SM: thread r of the epilogue owns
// accumulator row r, so direct global stores touch 32 different rows per warp instruction
// (uncoalesced, 32 L1 wavefronts each).  Here every 32-column fp32 slice / 64-column bf16 slice of
// the tile is written into a 128-row x 128-byte shared-memory box (SWIZZLE_128B pattern, conflict
// free) and moved by TMA:
//     residual:  global --TMA load--> box --(+ in place)--> box --TMA store--> global
// A dedicated "DMA" warp (warp 3: lane 0 = fp32 boxes, lane 1 = bf16 boxes) issues the bulk tensor
// copies; it talks to the 128 epilogue threads through mbarriers only.  TMA clips rows >= M,
// columns >= n_real and pixels outside the image, so the compute code has no bounds checks.
#include "gemm.cuh"

namespace hitsir {

namespace {

constexpr int kBoxBytes = 128 * 128;     // 128 rows x 128 B
constexpr int kNBox = 6;                 // box buffers shared by the fp32 and bf16 streams
// Epilogue warps: EQ per TMEM lane quarter (2 or 4), each handles a 64/EQ-column slice of every 64-column group.  EQ = 4 (16 warps)
// hides the TMEM-load / math / store latency chain of the activation epilogues; 64-column tiles keep EQ = 2.

template <int BN>
struct TmaCfg {
  static constexpr int kStages = (BN >= 160) ? 3 : 4;
  static constexpr int kABytes = 128 * 128;
  static constexpr int kBBytes = BN * 128;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kTmemCols = (2 * BN <= 32) ? 32 : (2 * BN <= 64) ? 64 : (2 * BN <= 128) ? 128 : (2 * BN <= 256) ? 256 : 512;
  static constexpr int kPipeBytes = kStages * kStageBytes;
  static constexpr int kMaxCols = (BN == 160) ? 960 : 384;   // bias staged in smem for every N tile (n_tiles * BN <= kMaxCols)
  static constexpr int kParamBytes = kMaxCols * 4;
  static constexpr int kSmemBytes = kPipeBytes + kNBox * kBoxBytes + kParamBytes + 1024 + 512;
  static constexpr int kGroups = BN / 64;       // 64-column output groups per tile (BN = 160: the 128 gated columns of EPI_MSGATE)
  static constexpr int kOutCols = kGroups * 64; // output columns produced per N tile
};

struct TileCoord {
  int m_tile, n_tile, b, y0, x0;
};
__device__ __forceinline__ TileCoord tile_coord(const GemmParams& p, int w) {
  TileCoord t;
  t.n_tile = w % p.n_tiles; t.m_tile = w / p.n_tiles;
  const ConvTile c = p.conv ? conv_tile(t.m_tile, p.tiles_x, p.tiles_y) : ConvTile{0, 0, 0};
  t.b = c.b; t.y0 = c.y0; t.x0 = c.x0;
  return t;
}

}  // namespace

static_assert(TmaCfg<160>::kSmemBytes <= 232448 && TmaCfg<192>::kSmemBytes <= 232448 && TmaCfg<64>::kSmemBytes <= 232448, "smem budget");

template <int BN, int EQ>
__global__ void __launch_bounds__(128 + 128 * EQ, 1)
umma_gemm_tma_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                     const __grid_constant__ CUtensorMap tmap_f, const __grid_constant__ CUtensorMap tmap_h,
                     const __grid_constant__ CUtensorMap tmap_r, const GemmParams p) {
  using Cfg = TmaCfg<BN>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_al = smem_raw + (smem_base - smem_u32(smem_raw));
  const bool has_f32 = p.out_f32 != nullptr;
  const bool has_b16 = p.out_bf16 != nullptr;
  const bool has_res = p.res != nullptr;
  // box buffers: the first nf belong to the fp32 stream, the remaining nh to the bf16 stream
  const int nf = has_f32 ? (has_b16 ? 4 : kNBox) : 0;
  const int nh = kNBox - nf;
  const uint32_t box0 = smem_base + Cfg::kPipeBytes;
  uint8_t* box_ptr = smem_al + Cfg::kPipeBytes;
  float* s_bias = reinterpret_cast<float*>(box_ptr + kNBox * kBoxBytes);
  constexpr int kMaxCols = Cfg::kMaxCols;
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_bias + kMaxCols);
  const uint32_t bar0 = smem_u32(bars);
  constexpr int S = Cfg::kStages;
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (S + s); };
  auto tfull_bar = [&](int s) { return bar0 + 8u * (2 * S + s); };
  auto tempty_bar = [&](int s) { return bar0 + 8u * (2 * S + 2 + s); };
  auto in_bar = [&](int s) { return bar0 + 8u * (2 * S + 4 + s); };              // DMA -> epilogue: box s usable (residual landed / free)
  auto out_bar = [&](int s) { return bar0 + 8u * (2 * S + 4 + kNBox + s); };     // epilogue -> DMA: box s written
  const uint32_t bres_full = bar0 + 8u * (2 * S + 4 + 2 * kNBox);                // resident-weights mode: the CTA's weight tile has landed
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 2 * S + 4 + 2 * kNBox + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int total = p.m_tiles * p.n_tiles;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    if (has_f32) tma_prefetch_desc(&tmap_f);
    if (has_b16) tma_prefetch_desc(&tmap_h);
    if (has_res) tma_prefetch_desc(&tmap_r);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < S; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(tfull_bar(s), 1); mbar_init(tempty_bar(s), 4 * EQ); }
    mbar_init(bres_full, 1);
    for (int s = 0; s < kNBox; ++s) {
      mbar_init(in_bar(s), 1);
      mbar_init(out_bar(s), s < nf ? 2 * EQ : 4 * EQ);   // warp-level arrivals; fp32 box (32 columns): half of the slices; bf16 box (64): all
    }
    fence_barrier_init();
  }
  if (warp == 2) {
    tmem_alloc(smem_u32(tmem_ptr_smem), Cfg::kTmemCols);
    tmem_relinquish();
  }
  {
    const int ncols = p.n_tiles * BN;
    for (int i = threadIdx.x; i < kMaxCols; i += blockDim.x) s_bias[i] = i < ncols ? p.bias[i] : 0.f;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  pdl_entry();                                           // up to here only weights (bias) were read

  if (warp == 0) {
    if (lane == 0) {
      // ===================== operand TMA producer =====================
      int stage = 0; uint32_t phase = 0;
      if (p.b_resident) {
        // Resident weights: every tile of this CTA has the same N tile (grid % n_tiles == 0), so its [BN x K] weight tile is fetched once
        // into the head of the pipeline area and only the A k-blocks cycle through the ring behind it.  Re-streaming the weights for
        // every 128-token tile made the linears L2->SM-bound (fc1: 240 KB per 128 tokens, DESIGN.md 3.3).
        const int n_tile = (int)(blockIdx.x % (unsigned)p.n_tiles);
        mbar_expect_tx(bres_full, p.num_kb * Cfg::kBBytes);
        for (int kb = 0; kb < p.num_kb; ++kb) tma_load_2d(smem_base + kb * Cfg::kBBytes, &tmap_b, bres_full, kb * 64, n_tile * BN);
        const uint32_t ring = smem_base + p.num_kb * Cfg::kBBytes;
        for (int w = blockIdx.x; w < total; w += gridDim.x) {
          const TileCoord t = tile_coord(p, w);
          for (int kb = 0; kb < p.num_kb; ++kb) {
            mbar_wait(empty_bar(stage), phase ^ 1u);
            mbar_expect_tx(full_bar(stage), Cfg::kABytes);
            tma_load_2d(ring + stage * Cfg::kABytes, &tmap_a, full_bar(stage), kb * 64, t.m_tile * 128);
            if (++stage == S) { stage = 0; phase ^= 1u; }
          }
        }
      } else
      for (int w = blockIdx.x; w < total; w += gridDim.x) {
        const TileCoord t = tile_coord(p, w);
        for (int kb = 0; kb < p.num_kb; ++kb) {
          mbar_wait(empty_bar(stage), phase ^ 1u);
          const uint32_t sa = smem_base + stage * Cfg::kStageBytes;
          const uint32_t sb = sa + Cfg::kABytes;
          mbar_expect_tx(full_bar(stage), Cfg::kStageBytes);
          if (p.conv) {
            const int tap = kb / p.cblocks, cb = kb - tap * p.cblocks;
            tma_load_4d(sa, &tmap_a, full_bar(stage), cb * 64, t.x0 + tap % 3 - 1, t.y0 + tap / 3 - 1 + p.a_y_off, t.b);
          } else {
            tma_load_2d(sa, &tmap_a, full_bar(stage), kb * 64, t.m_tile * 128);
          }
          tma_load_2d(sb, &tmap_b, full_bar(stage), kb * 64, t.n_tile * BN);
          if (++stage == S) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ===================== MMA issuer =====================
      constexpr uint32_t idesc = umma_idesc_bf16(128, BN);
      int stage = 0; uint32_t phase = 0;
      int it = 0;
      for (int w = blockIdx.x; w < total; w += gridDim.x, ++it) {
        const int as = it & 1;
        mbar_wait(tempty_bar(as), (((uint32_t)(it >> 1)) & 1u) ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(as * BN);
        if (p.b_resident && it == 0) mbar_wait(bres_full, 0u);
        for (int kb = 0; kb < p.num_kb; ++kb) {
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          const uint32_t sa = p.b_resident ? smem_base + p.num_kb * Cfg::kBBytes + stage * Cfg::kABytes : smem_base + stage * Cfg::kStageBytes;
          const uint64_t adesc = umma_desc_sw128(sa);
          const uint64_t bdesc = umma_desc_sw128(p.b_resident ? smem_base + kb * Cfg::kBBytes : sa + Cfg::kABytes);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (kb | k) != 0 ? 1u : 0u);
          umma_commit(empty_bar(stage));
          if (++stage == S) { stage = 0; phase ^= 1u; }
        }
        umma_commit(tfull_bar(as));
      }
    }
  } else if (warp == 3) {
    // ===================== epilogue DMA: lane 0 = fp32 boxes (+ residual loads), lane 1 = bf16 boxes ==========
    // Per tile the fp32 stream uses 2*kGroups boxes (32 columns each), the bf16 stream kGroups boxes (64 columns).
    const bool f_lane = (lane == 0 && has_f32), h_lane = (lane == 1 && has_b16);
    if (f_lane || h_lane) {
      const int nb = f_lane ? nf : nh;                 // ring size
      const int first = f_lane ? 0 : nf;               // first box buffer of this stream
      const int per_tile = f_lane ? 2 * Cfg::kGroups : Cfg::kGroups;
      const int width = f_lane ? 32 : 64;
      const int ncol_limit = f_lane ? p.n_real : p.ldb;
      const CUtensorMap* tm_out = f_lane ? &tmap_f : &tmap_h;
      int c0s[kNBox], r0s[kNBox], r1s[kNBox], r2s[kNBox];
      uint32_t u_prep = 0, u_store = 0;
      auto store_one = [&]() {
        const int s = (int)(u_store % (uint32_t)nb);
        const int b = first + s;
        mbar_wait(out_bar(b), (u_store / (uint32_t)nb) & 1u);
        if (c0s[s] < ncol_limit) {
          if (p.conv) tma_store_4d(tm_out, box0 + b * kBoxBytes, c0s[s], r0s[s], r1s[s], r2s[s]);
          else tma_store_2d(tm_out, box0 + b * kBoxBytes, c0s[s], r0s[s]);
          tma_commit();
        }
        ++u_store;
      };
      for (int w = blockIdx.x; w < total; w += gridDim.x) {
        const TileCoord t = tile_coord(p, w);
        for (int j = 0; j < per_tile; ++j) {
          const int col = t.n_tile * Cfg::kOutCols + width * j;
          const int s = (int)(u_prep % (uint32_t)nb);
          const int b = first + s;
          if (u_prep >= (uint32_t)nb) {
            // box s was last used by store #(u_prep - nb).  Bulk groups retire in order, so once the stores through #(u_prep - nb + 1)
            // are issued, "at most one group pending" proves that store has finished reading shared memory -- without waiting for the
            // newest store (waiting for group 0 here exposed one full store latency per box: ~6k cycles per fc1 tile).
            const uint32_t need = u_prep - (uint32_t)nb + 2u;
            while (u_store < need && u_store < u_prep) store_one();
            tma_wait_read<1>();
          }
          c0s[s] = col;
          if (p.conv) { r0s[s] = t.x0; r1s[s] = t.y0; r2s[s] = t.b; } else { r0s[s] = t.m_tile * 128; r1s[s] = 0; r2s[s] = 0; }
          if (f_lane && has_res && col < ncol_limit) {
            mbar_expect_tx(in_bar(b), kBoxBytes);
            if (p.conv) tma_load_4d(box0 + b * kBoxBytes, &tmap_r, in_bar(b), col, t.x0, t.y0, t.b);
            else tma_load_2d(box0 + b * kBoxBytes, &tmap_r, in_bar(b), col, t.m_tile * 128);
          } else {
            mbar_arrive(in_bar(b));
          }
          ++u_prep;
        }
      }
      while (u_store < u_prep) store_one();
      tma_wait_all0();
    }
  } else if (warp >= 4) {
    // ===================== epilogue compute (8 warps) =====================
    const int q = warp & 3;                            // TMEM lane quarter of this warp
    constexpr int SW = 64 / EQ;                        // slice width (columns) of one thread
    const int hs = (warp - 4) >> 2;                    // slice handled by this warp: columns 64g + SW*hs of every 64-column group g
    const int r = q * 32 + lane;
    const uint32_t rsw = (uint32_t)(r & 7);
    uint8_t* row_ptr = box_ptr + r * 128;              // this thread's row inside box 0
    auto ld_slice = [&](uint32_t taddr, float* v) {
      if constexpr (SW == 32) tmem_ld32(taddr, v); else tmem_ld16(taddr, v);
    };
    int it = 0;
    for (int w = blockIdx.x; w < total; w += gridDim.x, ++it) {
      const int n_tile = w % p.n_tiles;
      const int n0 = n_tile * BN;
      const int as = it & 1;
      mbar_wait(tfull_bar(as), ((uint32_t)(it >> 1)) & 1u);
      tc_fence_after();
      const uint32_t tacc = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * BN);
      float x1[SW];
      if (BN == 160 && p.epi == EPI_MSGATE) {
        // MultipleSizeConvExtract gate (hit_sir_pro.py:83-92): tile columns [32k, 32k+32), k = 0..3 hold conv3/5/7/9 of 32 embedding
        // channels, columns [128, 160) the 1x1 conv_x of the same channels; g_k = x_k * sigmoid(x_1 * x_k) + x_k
        const int ci0 = (SW * hs) & 31;
        ld_slice(tacc + 128 + ci0, x1);
#pragma unroll
        for (int i = 0; i < SW; ++i) x1[i] += s_bias[n0 + 128 + ci0 + i];
      }
#pragma unroll 1
      for (int g = 0; g < Cfg::kGroups; ++g) {
        const int c0 = 64 * g + SW * hs;               // tile-local first column of this thread's slice
        const int gc = n0 + c0;
        float v[SW];
        ld_slice(tacc + c0, v);
#pragma unroll
        for (int i = 0; i < SW; i += 4) {
          const float4 bb = *reinterpret_cast<const float4*>(s_bias + gc + i);
          v[i] += bb.x; v[i + 1] += bb.y; v[i + 2] += bb.z; v[i + 3] += bb.w;
        }
        if (BN == 160 && p.epi == EPI_MSGATE) {
#pragma unroll
          for (int i = 0; i < SW; ++i) {
            // x sigmoid(x1 x) + x with sigmoid(z) = rcp(1 + 2^(-z log2 e)): two MUFU ops instead of an exp and an IEEE division with its
            // range fix-ups (2.8 -> 1.6 ms at cfg2).  The one-MUFU tanh form used elsewhere is NOT good enough here: tanh.approx is
            // off by up to 2^-11 with a sign that follows the argument, the 768-term conv_last contraction adds those errors coherently,
            // and the error of the block0.4.scc tap doubled (5.1e-3 -> 1.2e-2) in the stress test.
            const float e = ex2_approx(-1.4426950408889634f * (x1[i] * v[i]));
            v[i] = fmaf(v[i], rcp_approx(1.0f + e), v[i]);
          }
        } else {
          if (p.act == ACT_LRELU) {
#pragma unroll
            for (int i = 0; i < SW; ++i) v[i] = lrelu(v[i], p.slope);
          }
          if (gc + SW > p.n_real) {
#pragma unroll
            for (int i = 0; i < SW; ++i) v[i] = (gc + i < p.n_real) ? v[i] : 0.f;
          }
        }
        if (has_f32) {
          // fp32 boxes hold 32 columns: box index 2g + (c0 % 64) / 32, this slice covers SW/4 of its 8 chunks
          const uint32_t u = (uint32_t)it * (uint32_t)(2 * Cfg::kGroups) + (uint32_t)(2 * g + ((SW * hs) >> 5));
          const int b = (int)(u % (uint32_t)nf);
          mbar_wait(in_bar(b), (u / (uint32_t)nf) & 1u);
          uint8_t* fb = row_ptr + b * kBoxBytes;
          const uint32_t ch0 = (uint32_t)(((SW * hs) & 31) >> 2);
#pragma unroll
          for (int ch = 0; ch < SW / 4; ++ch) {
            float4* ptr = reinterpret_cast<float4*>(fb + (((ch0 + (uint32_t)ch) ^ rsw) << 4));
            float4 o = make_float4(v[4 * ch], v[4 * ch + 1], v[4 * ch + 2], v[4 * ch + 3]);
            if (has_res) {
              const float4 rr = *ptr;
              o.x += rr.x; o.y += rr.y; o.z += rr.z; o.w += rr.w;
              v[4 * ch] = o.x; v[4 * ch + 1] = o.y; v[4 * ch + 2] = o.z; v[4 * ch + 3] = o.w;
            }
            *ptr = o;
          }
          fence_proxy_async_smem();
          mbar_arrive_warp(out_bar(b));
        }
        if (has_b16) {
          const uint32_t u = (uint32_t)it * (uint32_t)Cfg::kGroups + (uint32_t)g;
          const int b = nf + (int)(u % (uint32_t)nh);
          mbar_wait(in_bar(b), (u / (uint32_t)nh) & 1u);
          uint8_t* hb = row_ptr + b * kBoxBytes;
#pragma unroll
          for (int ch = 0; ch < SW / 8; ++ch) {
            uint4 o = make_uint4(pack_bf16x2(v[8 * ch], v[8 * ch + 1]), pack_bf16x2(v[8 * ch + 2], v[8 * ch + 3]),
                                 pack_bf16x2(v[8 * ch + 4], v[8 * ch + 5]), pack_bf16x2(v[8 * ch + 6], v[8 * ch + 7]));
            *reinterpret_cast<uint4*>(hb + (((uint32_t)((SW / 8) * hs + ch) ^ rsw) << 4)) = o;
          }
          fence_proxy_async_smem();
          mbar_arrive_warp(out_bar(b));
        }
      }
      tc_fence_before();
      mbar_arrive_warp(tempty_bar(as));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

template <int BN, int EQ>
static int launch_tma_bn(const GemmParams& p, const CUtensorMap* maps, int num_sms, cudaStream_t st) {
  using Cfg = TmaCfg<BN>;
  static unsigned long long configured = 0;
  if (ensure_dynamic_smem(umma_gemm_tma_kernel<BN, EQ>, Cfg::kSmemBytes, &configured)) return 1;
  const int total = p.m_tiles * p.n_tiles;
  const int grid = total < num_sms ? total : num_sms;
  if (grid <= 0) return 0;
  GemmParams q = p;
  q.b_resident = (p.b_resident && !p.conv && grid % p.n_tiles == 0 &&
                  p.num_kb * Cfg::kBBytes + Cfg::kStages * Cfg::kABytes <= Cfg::kPipeBytes) ? 1 : 0;
  if (p.n_tiles * BN > Cfg::kMaxCols) { set_error("launch_umma_gemm_tma: %d output columns exceed the staged-parameter limit %d", p.n_tiles * BN, Cfg::kMaxCols); return 1; }
  HITSIR_CHECK(launch_pdl(umma_gemm_tma_kernel<BN, EQ>, dim3(grid), dim3(128 + 128 * EQ), Cfg::kSmemBytes, st, maps[0], maps[1], maps[2], maps[3], maps[4], q));
  return 0;
}

// maps: {A, B, out_f32, out_bf16, residual}; unused maps may be copies of any valid map
int launch_umma_gemm_tma(int BN, const GemmParams& p, const CUtensorMap* maps, int num_sms, cudaStream_t st) {
  if (p.epi != EPI_STORE && p.epi != EPI_MSGATE) { set_error("launch_umma_gemm_tma: unsupported epilogue %d", p.epi); return 1; }
  switch (BN) {
    case 64: return launch_tma_bn<64, 2>(p, maps, num_sms, st);     // 64-column tiles: the 8-warp epilogue is already hidden under the 9-tap mainloop
    case 160: return launch_tma_bn<160, 4>(p, maps, num_sms, st);
    case 192: return launch_tma_bn<192, 4>(p, maps, num_sms, st);
    default: set_error("launch_umma_gemm_tma: unsupported N tile %d", BN); return 1;
  }
}

}  // namespace hitsir
