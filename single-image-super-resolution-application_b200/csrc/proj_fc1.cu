// proj + norm1 + residual and fc1 + GELU of one transformer block in one persistent tcgen05 kernel (hit_sir_pro.py:597, :700-703, :39-41):
//     x' = x + LN1(outsc Wp^T + bp)          -> fp32 stream (`xout`)
//     h1 = GELU(bf16(x') W1^T + b1)          -> bf16 [M, 384] (`h1`, columns 360..383 zero)
// bf16(x') is the fc1 A operand: the LayerNorm epilogue writes it straight into a 128B-swizzled K-major operand in shared memory, so the
// bf16 copy of the stream that the two separate linears exchanged through HBM (384 B per token, written and read back) never leaves the SM.
//
// Per 128-token tile the MMA issuer computes three [128 x 192] accumulators in order, D1 = proj, D2a / D2b = the two N = 192 halves of
// fc1, rotating over two TMEM regions: D1(i) -> R(3i % 2), D2a(i) -> the other, D2b(i) -> D1's region once the LayerNorm epilogue has
// released it, D1(i + 1) -> D2a's region once the GELU epilogue has released it.  So the MMAs of the next accumulator run while the
// epilogue works on the current one, and every HBM byte moves through TMA boxes issued by their own lanes:
//   warp 0: lane 0 loads the outsc k-blocks, lane 1 streams the weights from L2 as [192 N x 64 K] units (3 Wp + 6 W1 per tile)
//   warp 1: tcgen05.mma issuer;  warp 2: TMEM allocation
//   warp 3: lane 0 = epilogue boxes (residual in, stream out, h1 out)
//   warps 4..19: epilogue, 4 warps per TMEM lane quarter, each a 16-column slice of every 64-column group
// Results are bit-identical to the two-kernel chain (umma_gemm_tma.cu at BN = 192): same MMA shapes and k order, and the LayerNorm
// statistics are the 32-column-slice Chan partials merged in the order of the 8-warp LayerNorm epilogue (see below).
#include "gemm.cuh"
#include "kernels.cuh"

namespace hitsir {

namespace {

constexpr int kBox = 128 * 128;              // one 128-row x 128-byte box: a 64-column bf16 k-block or a 32-column fp32 slice
constexpr int kUnit = 192 * 128;             // one [192 N x 64 K] bf16 weight unit
constexpr int kNBox = 5;                     // epilogue boxes, used in turn by the fp32 stream (residual in, x' out) and h1 (out)
constexpr int kEpiWarps = 16;
constexpr int kOffW = 2 * kBox;              // outsc ring: 2 k-blocks
constexpr int kOffA2 = kOffW + 2 * kUnit;    // weight ring: 2 units
constexpr int kOffBox = kOffA2 + 3 * kBox;   // fc1 A operand: 3 k-blocks
constexpr int kOffPar = kOffBox + kNBox * kBox;
constexpr int kOffPart = kOffPar + (3 * 192 + 384) * 4;   // bp | gamma | beta | b1
constexpr int kOffBar = kOffPart + 2 * 2 * 128 * 8;       // LayerNorm partials [2 tile parity][2 column halves][128 rows]
constexpr int kNumBars = 13 + 2 * kNBox;
constexpr int kSmemBytes = kOffBar + kNumBars * 8 + 8 + 1024;
static_assert(kSmemBytes <= 232448, "smem budget");


}  // namespace

__global__ void __launch_bounds__(128 + 32 * kEpiWarps, 1)
proj_fc1_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_wp, const __grid_constant__ CUtensorMap tm_w1,
                const __grid_constant__ CUtensorMap tm_res, const __grid_constant__ CUtensorMap tm_out, const __grid_constant__ CUtensorMap tm_h1,
                const ProjFc1Params p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sm = smem_raw + (base - smem_u32(smem_raw));
  float* s_bp = reinterpret_cast<float*>(sm + kOffPar);
  float* s_g = s_bp + 192;
  float* s_be = s_g + 192;
  float* s_b1 = s_be + 192;
  float2* s_part = reinterpret_cast<float2*>(sm + kOffPart);
  const uint32_t bar0 = base + kOffBar;
  auto a_full = [&](int s) { return bar0 + 8u * s; };
  auto a_empty = [&](int s) { return bar0 + 8u * (2 + s); };
  auto w_full = [&](int s) { return bar0 + 8u * (4 + s); };
  auto w_empty = [&](int s) { return bar0 + 8u * (6 + s); };
  auto tfull = [&](int s) { return bar0 + 8u * (8 + s); };
  auto tempty = [&](int s) { return bar0 + 8u * (10 + s); };
  const uint32_t a2_full = bar0 + 8u * 12;                                   // epilogue -> MMA: the fc1 A operand of this tile is written
  auto in_bar = [&](int b) { return bar0 + 8u * (13 + b); };                 // DMA -> epilogue: box b usable (residual landed / free)
  auto out_bar = [&](int b) { return bar0 + 8u * (13 + kNBox + b); };        // epilogue -> DMA: box b written
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sm + kOffBar + kNumBars * 8);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_a); tma_prefetch_desc(&tm_wp); tma_prefetch_desc(&tm_w1);
    tma_prefetch_desc(&tm_res); tma_prefetch_desc(&tm_out); tma_prefetch_desc(&tm_h1);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < 2; ++s) {
      mbar_init(a_full(s), 1); mbar_init(a_empty(s), 1); mbar_init(w_full(s), 1); mbar_init(w_empty(s), 1);
      mbar_init(tfull(s), 1); mbar_init(tempty(s), kEpiWarps);
    }
    mbar_init(a2_full, kEpiWarps);
    for (int b = 0; b < kNBox; ++b) { mbar_init(in_bar(b), 1); mbar_init(out_bar(b), kEpiWarps); }
    fence_barrier_init();
  }
  if (warp == 2) {
    tmem_alloc(smem_u32(tmem_slot), 512);
    tmem_relinquish();
  }
  for (int i = threadIdx.x; i < 192; i += blockDim.x) {
    s_bp[i] = p.bias_p[i];
    s_g[i] = i < kC ? p.gamma[i] : 0.f;        // zero beyond 180: the pad columns of the stream and of bf16(x') become 0
    s_be[i] = i < kC ? p.beta[i] : 0.f;
  }
  for (int i = threadIdx.x; i < kHidp; i += blockDim.x) s_b1[i] = p.bias1[i];
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_entry();                                 // up to here only weights were read

  if (warp == 0) {
    if (lane == 0) {
      // ===================== outsc k-blocks =====================
      int s = 0; uint32_t ph = 0;
      for (int w = blockIdx.x; w < p.m_tiles; w += gridDim.x)
        for (int kb = 0; kb < 3; ++kb) {
          mbar_wait_park(a_empty(s), ph ^ 1u);
          mbar_expect_tx(a_full(s), kBox);
          tma_load_2d(base + s * kBox, &tm_a, a_full(s), kb * 64, w * 128);
          if (++s == 2) { s = 0; ph ^= 1u; }
        }
    } else if (lane == 1) {
      // ===================== weight units: Wp k-blocks 0..2, then W1 rows [192 h, 192 h + 192) k-blocks 0..2 for h = 0, 1 ===========
      int s = 0; uint32_t ph = 0;
      for (int w = blockIdx.x; w < p.m_tiles; w += gridDim.x)
        for (int u = 0; u < 9; ++u) {
          mbar_wait_park(w_empty(s), ph ^ 1u);
          mbar_expect_tx(w_full(s), kUnit);
          const uint32_t dst = base + kOffW + s * kUnit;
          if (u < 3) tma_load_2d(dst, &tm_wp, w_full(s), u * 64, 0);
          else tma_load_2d(dst, &tm_w1, w_full(s), ((u - 3) % 3) * 64, ((u - 3) / 3) * 192);
          if (++s == 2) { s = 0; ph ^= 1u; }
        }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ===================== MMA issuer =====================
      constexpr uint32_t idesc = umma_idesc_bf16(128, 192);
      int as = 0, ws = 0; uint32_t aph = 0, wph = 0, ac = 0;
      int it = 0;
      for (int w = blockIdx.x; w < p.m_tiles; w += gridDim.x, ++it) {
        for (int m = 0; m < 3; ++m, ++ac) {    // m = 0: proj, 1 / 2: fc1 halves
          const uint32_t reg = ac & 1u;
          mbar_wait_park(tempty(reg), ((ac >> 1) & 1u) ^ 1u);
          if (m == 1) mbar_wait_park(a2_full, (uint32_t)it & 1u);
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + reg * 192u;
          for (int kb = 0; kb < 3; ++kb) {
            if (m == 0) mbar_wait_park(a_full(as), aph);
            mbar_wait_park(w_full(ws), wph);
            tc_fence_after();
            const uint64_t adesc = umma_desc_sw128(m == 0 ? base + as * kBox : base + kOffA2 + kb * kBox);
            const uint64_t bdesc = umma_desc_sw128(base + kOffW + ws * kUnit);
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_bf16(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (kb | k) != 0 ? 1u : 0u);
            umma_commit(w_empty(ws));
            if (++ws == 2) { ws = 0; wph ^= 1u; }
            if (m == 0) {
              umma_commit(a_empty(as));
              if (++as == 2) { as = 0; aph ^= 1u; }
            }
          }
          umma_commit(tfull(reg));
        }
      }
    }
  } else if (warp == 3) {
    // ===================== epilogue DMA =====================
    // Per tile twelve box uses in the order the epilogue fills them: six 32-column fp32 boxes of x' (residual loaded first; columns
    // >= 180 are clipped by TMA), then six 64-column bf16 boxes of h1.  The two kinds never overlap in time inside the epilogue, so one
    // ring serves both and each phase runs with all kNBox boxes in flight.
    if (lane == 0) {
      uint32_t u_prep = 0, u_store = 0;
      auto is_f32 = [](uint32_t u) { return u % 12u < 6u; };
      auto box_col = [](uint32_t u) { const int j = (int)(u % 12u); return j < 6 ? 32 * j : 64 * (j - 6); };
      auto box_row = [&](uint32_t u) { return ((int)blockIdx.x + (int)(u / 12u) * (int)gridDim.x) * 128; };
      auto store_one = [&]() {
        const int b = (int)(u_store % (uint32_t)kNBox);
        mbar_wait_park(out_bar(b), (u_store / (uint32_t)kNBox) & 1u);
        tma_store_2d(is_f32(u_store) ? &tm_out : &tm_h1, base + kOffBox + b * kBox, box_col(u_store), box_row(u_store));
        tma_commit();
        ++u_store;
      };
      for (int w = blockIdx.x; w < p.m_tiles; w += gridDim.x) {
        for (int j = 0; j < 12; ++j) {
          const int b = (int)(u_prep % (uint32_t)kNBox);
          if (u_prep >= (uint32_t)kNBox) {
            // box b was last used by store #(u_prep - kNBox).  Bulk groups retire in order, so once the stores through
            // #(u_prep - kNBox + 1) are issued, "at most one group pending" proves that store has finished reading shared memory.
            const uint32_t need = u_prep - (uint32_t)kNBox + 2u;
            while (u_store < need && u_store < u_prep) store_one();
            tma_wait_read<1>();
          }
          if (is_f32(u_prep)) {
            mbar_expect_tx(in_bar(b), kBox);
            tma_load_2d(base + kOffBox + b * kBox, &tm_res, in_bar(b), box_col(u_prep), w * 128);
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
    // ===================== epilogue (16 warps) =====================
    const int q = warp & 3;                    // TMEM lane quarter of this warp
    const int hs = (warp - 4) >> 2;            // 16-column slice: columns 64 g + 16 hs of every 64-column group g
    const int r = q * 32 + lane;
    const uint32_t rsw = (uint32_t)(r & 7);
    uint8_t* row_ptr = sm + kOffBox + r * 128;
    uint8_t* a2_row = sm + kOffA2 + r * 128;
    uint32_t ac = 0;
    int it = 0;
    for (int w = blockIdx.x; w < p.m_tiles; w += gridDim.x, ++it) {
      // ---------- proj: x' = x + LN1(D1 + bp) -> fp32 boxes and the fc1 A operand ----------
      {
        const uint32_t reg = ac & 1u;
        mbar_wait(tfull(reg), (ac >> 1) & 1u);
        tc_fence_after();
        const uint32_t tacc = tmem_base + ((uint32_t)(q * 32) << 16) + reg * 192u;
        // LayerNorm statistics without cancellation: per 32-column slice (mean, M2), merged with Chan's parallel update.  Warps hs = 0, 1
        // compute the partial of column half hs (columns 64 g + 32 hs, g = 0..2) exactly as the 8-warp epilogue of umma_gemm_tma.cu did;
        // each warp then starts from the partial of the half its own columns lie in and merges the other one, the order that epilogue
        // used for those columns.  So mean and rstd, and with them the stream, are bit-identical to the unfused proj.
        auto slice_count = [&](int ho) {
          int cn = 0;
          for (int g = 0; g < 3; ++g) cn += min(32, max(0, kC - (64 * g + 32 * ho)));
          return cn;
        };
        float2* part = s_part + (it & 1) * 256;
        if (hs < 2) {
          float n = 0.f, mean = 0.f, m2 = 0.f;
#pragma unroll 1
          for (int g = 0; g < 3; ++g) {
            const int c0 = 64 * g + 32 * hs;
            float v[32];
            tmem_ld32(tacc + c0, v);
            const int cnt = min(32, max(0, kC - c0));
            float sg = 0.f, qg = 0.f, mg;
            if (cnt == 32) {
#pragma unroll
              for (int i = 0; i < 32; ++i) { v[i] += s_bp[c0 + i]; sg += v[i]; }
              mg = sg * (1.0f / 32.0f);
#pragma unroll
              for (int i = 0; i < 32; ++i) { const float d = v[i] - mg; qg = fmaf(d, d, qg); }
            } else {
#pragma unroll
              for (int i = 0; i < 32; ++i) { v[i] += s_bp[c0 + i]; if (i < cnt) sg += v[i]; }
              mg = sg / (float)max(cnt, 1);
#pragma unroll
              for (int i = 0; i < 32; ++i) { const float d = v[i] - mg; if (i < cnt) qg = fmaf(d, d, qg); }
            }
            if (cnt > 0) {
              const float nn = n + (float)cnt, d = mg - mean;
              mean += d * ((float)cnt / nn);
              m2 += qg + d * d * (n * (float)cnt / nn);
              n = nn;
            }
          }
          part[hs * 128 + r] = make_float2(mean, m2);
        }
        named_bar_sync(1, 32 * kEpiWarps);   // the epilogue threads only
        const int h0 = hs >> 1, ho = h0 ^ 1;   // column half of this warp's slices, and the other half
        const float2 own = part[h0 * 128 + r];
        float n = (float)slice_count(h0), mean = own.x, m2 = own.y;
        {
          const float cnt = (float)slice_count(ho);
          if (cnt > 0.f) {
            const float2 t = part[ho * 128 + r];
            const float nn = n + cnt, d = t.x - mean;
            mean += d * (cnt / nn);
            m2 += t.y + d * d * (n * cnt / nn);
          }
        }
        const float rstd = rsqrtf(m2 / (float)kC + 1e-5f);
#pragma unroll 1
        for (int g = 0; g < 3; ++g) {
          const int c0 = 64 * g + 16 * hs;
          float v[16];
          tmem_ld16(tacc + c0, v);
#pragma unroll
          for (int i = 0; i < 16; i += 4) {
            const float4 bb = *reinterpret_cast<const float4*>(s_bp + c0 + i);
            v[i] += bb.x; v[i + 1] += bb.y; v[i + 2] += bb.z; v[i + 3] += bb.w;
          }
#pragma unroll
          for (int i = 0; i < 16; i += 4) {
            const float4 gg = *reinterpret_cast<const float4*>(s_g + c0 + i);
            const float4 be = *reinterpret_cast<const float4*>(s_be + c0 + i);
            v[i] = fmaf((v[i] - mean) * rstd, gg.x, be.x);
            v[i + 1] = fmaf((v[i + 1] - mean) * rstd, gg.y, be.y);
            v[i + 2] = fmaf((v[i + 2] - mean) * rstd, gg.z, be.z);
            v[i + 3] = fmaf((v[i + 3] - mean) * rstd, gg.w, be.w);
          }
          // fp32 box 2g + hs / 2 (32 columns), this slice is 4 of its 8 chunks: + residual in place.  Every warp arrives on both boxes of
          // the group (each box counts all 16 warps, as an h1 box does); it waits for the partner box to be handed out before arriving,
          // so the arrival cannot fall into the box's previous phase.
          const uint32_t u0 = (uint32_t)it * 12u + (uint32_t)(2 * g);
          const uint32_t u = u0 + (uint32_t)(hs >> 1), up = u ^ 1u;
          const int b = (int)(u % (uint32_t)kNBox), bp = (int)(up % (uint32_t)kNBox);
          mbar_wait(in_bar(b), (u / (uint32_t)kNBox) & 1u);
          uint8_t* fb = row_ptr + b * kBox;
          const uint32_t ch0 = (uint32_t)((hs & 1) * 4);
#pragma unroll
          for (int ch = 0; ch < 4; ++ch) {
            float4* ptr = reinterpret_cast<float4*>(fb + (((ch0 + (uint32_t)ch) ^ rsw) << 4));
            const float4 rr = *ptr;
            const float4 o = make_float4(v[4 * ch] + rr.x, v[4 * ch + 1] + rr.y, v[4 * ch + 2] + rr.z, v[4 * ch + 3] + rr.w);
            v[4 * ch] = o.x; v[4 * ch + 1] = o.y; v[4 * ch + 2] = o.z; v[4 * ch + 3] = o.w;
            *ptr = o;
          }
          fence_proxy_async_smem();
          mbar_arrive_warp(out_bar(b));
          mbar_wait(in_bar(bp), (up / (uint32_t)kNBox) & 1u);
          mbar_arrive_warp(out_bar(bp));
          // bf16(x') into k-block g of the fc1 A operand (the byte image of a SWIZZLE_128B box): chunks 2 hs, 2 hs + 1 of row r
#pragma unroll
          for (int ch = 0; ch < 2; ++ch) {
            const uint4 o = make_uint4(pack_bf16x2(v[8 * ch], v[8 * ch + 1]), pack_bf16x2(v[8 * ch + 2], v[8 * ch + 3]),
                                       pack_bf16x2(v[8 * ch + 4], v[8 * ch + 5]), pack_bf16x2(v[8 * ch + 6], v[8 * ch + 7]));
            *reinterpret_cast<uint4*>(a2_row + g * kBox + (((uint32_t)(2 * hs + ch) ^ rsw) << 4)) = o;
          }
        }
        fence_proxy_async_smem();
        tc_fence_before();
        mbar_arrive_warp(tempty(reg));
        mbar_arrive_warp(a2_full);
        ++ac;
      }
      // ---------- fc1 halves: h1[:, 192 h + c] = GELU(D2 + b1), zero beyond column 360 ----------
#pragma unroll 1
      for (int h = 0; h < 2; ++h, ++ac) {
        const uint32_t reg = ac & 1u;
        mbar_wait(tfull(reg), (ac >> 1) & 1u);
        tc_fence_after();
        const uint32_t tacc = tmem_base + ((uint32_t)(q * 32) << 16) + reg * 192u;
#pragma unroll 1
        for (int g = 0; g < 3; ++g) {
          const int c0 = 64 * g + 16 * hs;
          const int gc = 192 * h + c0;
          float v[16];
          tmem_ld16(tacc + c0, v);
#pragma unroll
          for (int i = 0; i < 16; i += 4) {
            const float4 bb = *reinterpret_cast<const float4*>(s_b1 + gc + i);
            v[i] += bb.x; v[i + 1] += bb.y; v[i + 2] += bb.z; v[i + 3] += bb.w;
          }
#pragma unroll
          for (int i = 0; i < 16; i += 2) { const float2 gl = gelu2(make_float2(v[i], v[i + 1])); v[i] = gl.x; v[i + 1] = gl.y; }
          if (gc + 16 > kHid) {
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = (gc + i < kHid) ? v[i] : 0.f;
          }
          const uint32_t u = (uint32_t)it * 12u + 6u + (uint32_t)(3 * h + g);
          const int b = (int)(u % (uint32_t)kNBox);
          mbar_wait(in_bar(b), (u / (uint32_t)kNBox) & 1u);
          uint8_t* hb = row_ptr + b * kBox;
#pragma unroll
          for (int ch = 0; ch < 2; ++ch) {
            const uint4 o = make_uint4(pack_bf16x2(v[8 * ch], v[8 * ch + 1]), pack_bf16x2(v[8 * ch + 2], v[8 * ch + 3]),
                                       pack_bf16x2(v[8 * ch + 4], v[8 * ch + 5]), pack_bf16x2(v[8 * ch + 6], v[8 * ch + 7]));
            *reinterpret_cast<uint4*>(hb + (((uint32_t)(2 * hs + ch) ^ rsw) << 4)) = o;
          }
          fence_proxy_async_smem();
          mbar_arrive_warp(out_bar(b));
        }
        tc_fence_before();
        mbar_arrive_warp(tempty(reg));
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

int launch_proj_fc1(const ProjFc1Params& p, const CUtensorMap* maps, int num_sms, cudaStream_t st) {
  static unsigned long long configured = 0;
  if (ensure_dynamic_smem(proj_fc1_kernel, kSmemBytes, &configured)) return 1;
  const int grid = p.m_tiles < num_sms ? p.m_tiles : num_sms;
  if (grid <= 0) return 0;
  HITSIR_CHECK(launch_pdl(proj_fc1_kernel, dim3(grid), dim3(128 + 32 * kEpiWarps), kSmemBytes, st, maps[0], maps[1], maps[2], maps[3], maps[4], maps[5], p));
  return 0;
}

}  // namespace hitsir
