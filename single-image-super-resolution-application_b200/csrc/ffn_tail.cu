// Second half of ConvFFN fused into one persistent kernel (/root/reference/models/hit_sir_pro.py:42-46 with :15-17, and the
// post-norm residual of HierarchicalTransformerBlock.forward :704):
//     h2 = h1 + GELU(dwconv5x5(h1) + b_dw)            (warp-level bf16 MMAs with block-diagonal taps + packed-fp32 GELU)
//     x  = x + LayerNorm(h2 W2^T + b2)                 (tcgen05, accumulator in TMEM, LayerNorm in the epilogue)
// The 360-channel hidden map h2 never goes to HBM: per 8 x 16 pixel tile the conv warps produce it 64 channels at a time straight
// into the SWIZZLE_128B K-major A-operand buffers of the fc2 contraction, while the TMA producer streams the (8+4) x (16+4) x 64
// halo boxes of h1 (zero padding = out-of-bounds fill) and the matching 64-column slices of W2.  Standalone, the depthwise conv
// wrote and fc2 re-read 1536 B per token and fc2 sat at the HBM roofline; fused, fc2's traffic hides under the conv.
//
// The depthwise conv is a tensor-core contraction: an FP32-pipe version (25 FFMA per output, 3 distinct 64-bit operands per FFMA2 =
// 3 issue cycles, tools/ubench/ffma2_rate.cu) bound the kernel at 2.2-2.4 ms; m16n8k16 MMAs with B = diag(tap weights) waste 90 % of
// their flops and still run the 25 taps of 16 pixels x 8 channels in 13 instructions.
//
// Warp roles (640 threads): 0 = TMA producer, 1 = MMA issuer, 2 = TMEM allocator / statistics, 3 = residual/output box DMA,
// 4..19 = compute.  All 16 compute warps work on the same 64-channel slice (warp = 8 channels x 4 output rows of the tile); halo stage,
// A buffer and W2 stage ping-pong with the slice parity, so the next slice's halo is in flight while this one is convolved.  After every
// second slice the same warps run one 64-column group of the PREVIOUS tile's LayerNorm epilogue (warp = TMEM lane quarter x 16-column slice).
#include "gemm.cuh"
#include "kernels.cuh"

namespace hitsir {

namespace {

constexpr int kPH = 12, kPW = 20;                         // halo patch of an 8 x 16 tile
constexpr int kHalo = kPH * kPW * 128;                    // 30720 B, dense 128-byte pixel rows (no swizzle)
constexpr int kDwRow = 28;                                // words per channel of the tap table (kernels.cuh launch_pack_dw_mma)
constexpr int kDwTbl = 64 * kDwRow * 4;                   // the slice's 64 channel rows
constexpr int kHaloStage = 37 * 1024;                     // halo box + tap table, padded to keep the next region 1024-byte aligned
static_assert(kHalo + kDwTbl <= kHaloStage, "halo stage");
constexpr int kABuf = 128 * 128;                          // A operand: 128 pixels x 64 ch bf16, SWIZZLE_128B
constexpr int kWStage = 192 * 128;                        // W2 slice: 192 rows x 64 k
constexpr int kBoxBytes = 128 * 128;
constexpr int kNBox = 3;
constexpr int kOffHalo = 0;
constexpr int kOffA = 2 * kHaloStage;
constexpr int kOffWs = kOffA + 2 * kABuf;
constexpr int kOffBox = kOffWs + 2 * kWStage;
constexpr int kOffPar = kOffBox + kNBox * kBoxBytes;      // bias | gamma | beta (3 x 192 fp32)
constexpr int kOffPart = kOffPar + 3 * 192 * 4;           // LayerNorm partials [2][4][128] float2
constexpr int kOffPart2 = kOffPart + 2 * 4 * 128 * 8;      // per-pixel channel (sum, max) partials [4][128] float2
constexpr int kOffMult = kOffPart2 + 2 * 4 * 128 * 8;     // (double-buffered by tile parity); reflect multiplicity of the tile's 128 pixels (0 = outside the image)
constexpr int kOffZero = kOffMult + 128 * 4;                // 128 zero bytes: the tap row of the lanes whose B-fragment words are off-diagonal
constexpr int kOffBars = kOffZero + 128;
constexpr int kNumBars = 40;
constexpr int kSmemBytes = kOffBars + kNumBars * 8 + 16 + 1024;
static_assert(kSmemBytes <= 232448, "smem budget");
static_assert(kOffA % 1024 == 0 && kOffWs % 1024 == 0 && kOffBox % 1024 == 0, "swizzled regions need 1024-byte alignment");

struct Params {
  int B, H, W, tiles_x, tiles_y, total;
  const float* bias;        // fc2 bias [192] (zero padded)
  const float* gamma; const float* beta;     // norm2 [180]
  // casa statistics of the block output for the next block (SpatialChannelAttention :345-349), all optional (nullptr = off):
  float* cavg; float* cmax;                  // per pixel channel mean / max, [B*H*W]
  float* part_sum; float* part_max;          // per tile per channel: reflect-weighted sum / max over the tile's pixels, [total][180]
  int Hp, Wp;                                // reflect-padded size of the NEXT block's window grid
  const uint32_t* dw_tbl;                    // tap rows [384][28] (launch_pack_dw_mma)
  const uint8_t* w2_img;                     // fc2 weights as six SWIZZLE_128B operand images [192 rows x 64 k] (launch_pack_w2_image)
  bf16* shadow;                              // optional bf16 copy of the updated stream [B*H*W][192] (pads 0) for the RHTB conv that follows (:934)
  // band mode (exact multi-GPU sharding of one frame by rows, engine.cu): the h1 map has h1_y_off valid halo rows above row 0, and the
  // reflect multiplicities of the casa pools are those of the whole frame (row yg0 + y of a frame with Hf rows)
  int h1_y_off, yg0, Hf;
};

__device__ __forceinline__ void ldmatrix_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr) : "memory");
}
__device__ __forceinline__ void ldmatrix_x2(uint32_t addr, uint32_t& r0, uint32_t& r1) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0,%1}, [%2];" : "=r"(r0), "=r"(r1) : "r"(addr) : "memory");
}

__global__ void __launch_bounds__(640, 1)
ffn_tail_kernel(const __grid_constant__ CUtensorMap tm_h1, const __grid_constant__ CUtensorMap tm_x, const Params p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sb = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sp = smem_raw + (sb - smem_u32(smem_raw));
  float* s_bias = reinterpret_cast<float*>(sp + kOffPar);
  float* s_gamma = s_bias + 192;
  float* s_beta = s_gamma + 192;
  float2* s_part = reinterpret_cast<float2*>(sp + kOffPart);
  float2* s_part2 = reinterpret_cast<float2*>(sp + kOffPart2);
  float* s_mult = reinterpret_cast<float*>(sp + kOffMult);
  const bool want_stats = p.cavg != nullptr;
  const bool want_shadow = p.shadow != nullptr;
  const uint32_t bar0 = sb + kOffBars;
  auto halo_full = [&](int h) { return bar0 + 8u * h; };
  auto halo_empty = [&](int h) { return bar0 + 8u * (2 + h); };
  auto a_full = [&](int h) { return bar0 + 8u * (4 + h); };
  auto a_empty = [&](int h) { return bar0 + 8u * (6 + h); };
  auto w_full = [&](int h) { return bar0 + 8u * (8 + h); };
  auto w_empty = [&](int h) { return bar0 + 8u * (10 + h); };
  auto d_full = [&](int s) { return bar0 + 8u * (12 + s); };
  auto d_empty = [&](int s) { return bar0 + 8u * (14 + s); };
  auto in_bar = [&](int s) { return bar0 + 8u * (16 + s); };
  auto out_bar = [&](int s) { return bar0 + 8u * (16 + kNBox + s); };
  auto red_done = [&](int s) { return bar0 + 8u * (16 + 2 * kNBox + s); };      // statistics warp -> DMA: box s has been reduced
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(sp + kOffBars + kNumBars * 8);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) { tma_prefetch_desc(&tm_h1); tma_prefetch_desc(&tm_x); }
  if (warp == 1 && lane == 0) {
    for (int h = 0; h < 2; ++h) {
      mbar_init(halo_full(h), 1); mbar_init(halo_empty(h), 16);
      mbar_init(a_full(h), 16); mbar_init(a_empty(h), 1);
      mbar_init(w_full(h), 1); mbar_init(w_empty(h), 1);
      mbar_init(d_full(h), 1); mbar_init(d_empty(h), 16);
    }
    for (int s = 0; s < kNBox; ++s) { mbar_init(in_bar(s), 1); mbar_init(out_bar(s), 8); mbar_init(red_done(s), 1); }   // a 32-column box is written by 2 slices x 4 quarters
    fence_barrier_init();
  }
  if (warp == 2) { tmem_alloc(smem_u32(tmem_ptr_smem), 512); tmem_relinquish(); }   // warp 2 later doubles as the statistics warp
  if (threadIdx.x < 32) reinterpret_cast<uint32_t*>(sp + kOffZero)[threadIdx.x] = 0u;
  for (int i = threadIdx.x; i < 192; i += blockDim.x) {
    s_bias[i] = p.bias[i];
    s_gamma[i] = i < kC ? p.gamma[i] : 0.f;
    s_beta[i] = i < kC ? p.beta[i] : 0.f;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  pdl_entry();                                           // up to here only weights (fc2 bias, norm2) were read

  if (warp == 0) {
    if (lane == 0) {
      // ===================== producer: per 64-channel slice one h1 halo box and one W2 slice =====================
      int it = 0;
      for (int t = blockIdx.x; t < p.total; t += gridDim.x, ++it) {
        const auto [b, y0, x0] = conv_tile(t, p.tiles_x, p.tiles_y);
        for (int k = 0; k < 6; ++k) {
          const int h = k & 1;
          const uint32_t u = (uint32_t)(it * 3 + (k >> 1));
          mbar_wait_park(halo_empty(h), (u & 1u) ^ 1u);
          mbar_expect_tx(halo_full(h), kHalo + kDwTbl);
          tma_load_4d(sb + kOffHalo + h * kHaloStage, &tm_h1, halo_full(h), k * 64, x0 - 2, y0 - 2 + p.h1_y_off, b);
          bulk_load(sb + kOffHalo + h * kHaloStage + kHalo, p.dw_tbl + (size_t)k * (kDwTbl / 4), kDwTbl, halo_full(h));   // 64 contiguous tap rows
          mbar_wait_park(w_empty(h), (u & 1u) ^ 1u);
          mbar_expect_tx(w_full(h), kWStage);
          bulk_load(sb + kOffWs + h * kWStage, p.w2_img + (size_t)k * kWStage, kWStage, w_full(h));   // pre-swizzled operand image: one request, not 192 rows
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ===================== MMA issuer: D[128 x 192] += H2_slice[128 x 64] W2_slice^T =====================
      constexpr uint32_t idesc = umma_idesc_bf16(128, 192);
      int it = 0;
      for (int t = blockIdx.x; t < p.total; t += gridDim.x, ++it) {
        const int as = it & 1;
        mbar_wait_park(d_empty(as), (((uint32_t)(it >> 1)) & 1u) ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(as * 192);
        for (int k = 0; k < 6; ++k) {
          const int h = k & 1;
          const uint32_t u = (uint32_t)(it * 3 + (k >> 1));
          mbar_wait_park(a_full(h), u & 1u);
          mbar_wait_park(w_full(h), u & 1u);
          tc_fence_after();
          const uint64_t adesc = umma_desc_sw128(sb + kOffA + h * kABuf);
          const uint64_t bdesc = umma_desc_sw128(sb + kOffWs + h * kWStage);
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) umma_bf16(d_tmem, adesc + (uint64_t)(2 * kk), bdesc + (uint64_t)(2 * kk), idesc, (k | kk) != 0 ? 1u : 0u);
          umma_commit(a_empty(h));
          umma_commit(w_empty(h));
        }
        umma_commit(d_full(as));
      }
    }
  } else if (warp == 2) {
    // ===================== statistics warp (only with casa statistics on): reflect-weighted channel sums / maxima of every finished
    // 32-column box over its 128 pixels, for the next block's global pools.  lane = (row phase lane >> 3, 16-byte chunk lane & 7).
    if (want_stats) {
      uint32_t u = 0;
      for (int t = blockIdx.x; t < p.total; t += gridDim.x) {
        const auto [b, y0, x0] = conv_tile(t, p.tiles_x, p.tiles_y);
        for (int rr = lane; rr < 128; rr += 32) {
          const int y = y0 + (rr >> 4), x = x0 + (rr & 15);
          s_mult[rr] = (y < p.H && x < p.W) ? (float)(reflect_mult(y + p.yg0, p.Hf, p.Hp) * reflect_mult(x, p.W, p.Wp)) : 0.f;
        }
        __syncwarp();
        for (int j = 0; j < 6; ++j, ++u) {
          const int s = (int)(u % kNBox);
          mbar_wait_park(out_bar(s), (u / kNBox) & 1u);
          const uint8_t* box = sp + kOffBox + s * kBoxBytes;
          const int ck = lane & 7, rph = lane >> 3;
          float4 sum = make_float4(0.f, 0.f, 0.f, 0.f), mx = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
#pragma unroll 4
          for (int r4 = 0; r4 < 128; r4 += 4) {
            const int rr = r4 + rph;
            const float m = s_mult[rr];
            const float4 v = *reinterpret_cast<const float4*>(box + rr * 128 + (((uint32_t)ck ^ (uint32_t)(rr & 7)) << 4));
            sum.x = fmaf(m, v.x, sum.x); sum.y = fmaf(m, v.y, sum.y); sum.z = fmaf(m, v.z, sum.z); sum.w = fmaf(m, v.w, sum.w);
            if (m > 0.f) { mx.x = fmaxf(mx.x, v.x); mx.y = fmaxf(mx.y, v.y); mx.z = fmaxf(mx.z, v.z); mx.w = fmaxf(mx.w, v.w); }
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(red_done(s));          // every lane has read the box: it may be recycled once its store has drained too
#pragma unroll
          for (int o = 8; o <= 16; o <<= 1) {              // fixed-order merge of the four row phases: deterministic
            sum.x += __shfl_xor_sync(0xffffffffu, sum.x, o); sum.y += __shfl_xor_sync(0xffffffffu, sum.y, o);
            sum.z += __shfl_xor_sync(0xffffffffu, sum.z, o); sum.w += __shfl_xor_sync(0xffffffffu, sum.w, o);
            mx.x = fmaxf(mx.x, __shfl_xor_sync(0xffffffffu, mx.x, o)); mx.y = fmaxf(mx.y, __shfl_xor_sync(0xffffffffu, mx.y, o));
            mx.z = fmaxf(mx.z, __shfl_xor_sync(0xffffffffu, mx.z, o)); mx.w = fmaxf(mx.w, __shfl_xor_sync(0xffffffffu, mx.w, o));
          }
          const int col = 32 * j + 4 * ck;
          if (rph == 0 && col < kC) {                      // 180 = 45 chunks: a chunk is entirely real or entirely padding
            *reinterpret_cast<float4*>(p.part_sum + (long long)t * kC + col) = sum;
            *reinterpret_cast<float4*>(p.part_max + (long long)t * kC + col) = mx;
          }
        }
        __syncwarp();                                       // s_mult is rewritten for the next tile
      }
    } else if (want_shadow) {
      // the last block of a layer: no statistics are wanted, the warp converts every finished box to bf16 instead (16-byte chunks of 8
      // channels straight to global), which used to be a separate pass over the stream (cast_rows_bf16)
      uint32_t u = 0;
      for (int t = blockIdx.x; t < p.total; t += gridDim.x) {
        const auto [b, y0, x0] = conv_tile(t, p.tiles_x, p.tiles_y);
        for (int j = 0; j < 6; ++j, ++u) {
          const int s = (int)(u % kNBox);
          mbar_wait_park(out_bar(s), (u / kNBox) & 1u);
          const uint8_t* box = sp + kOffBox + s * kBoxBytes;
#pragma unroll 4
          for (int i = lane; i < 512; i += 32) {            // 128 pixels x 4 chunks of 8 channels
            const int rr = i >> 2, c8 = i & 3;
            const int y = y0 + (rr >> 4), x = x0 + (rr & 15);
            const float4 v0 = *reinterpret_cast<const float4*>(box + rr * 128 + (((uint32_t)(2 * c8) ^ (uint32_t)(rr & 7)) << 4));
            const float4 v1 = *reinterpret_cast<const float4*>(box + rr * 128 + (((uint32_t)(2 * c8 + 1) ^ (uint32_t)(rr & 7)) << 4));
            if (y < p.H && x < p.W)
              *reinterpret_cast<uint4*>(p.shadow + (((long long)b * p.H + y) * p.W + x) * kCp + 32 * j + 8 * c8) =
                  make_uint4(pack_bf16x2(v0.x, v0.y), pack_bf16x2(v0.z, v0.w), pack_bf16x2(v1.x, v1.y), pack_bf16x2(v1.z, v1.w));
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(red_done(s));
        }
      }
    }
  } else if (warp == 3) {
    if (lane == 0) {
      // ===================== box DMA: residual in, updated stream out (6 boxes of 32 fp32 columns per tile) =====================
      int c0s[kNBox], r0s[kNBox], r1s[kNBox], r2s[kNBox];
      uint32_t u_prep = 0, u_store = 0;
      auto store_one = [&]() {
        const int s = (int)(u_store % kNBox);
        mbar_wait_park(out_bar(s), (u_store / kNBox) & 1u);
        tma_store_4d(&tm_x, sb + kOffBox + s * kBoxBytes, c0s[s], r0s[s], r1s[s], r2s[s]);
        tma_commit();
        ++u_store;
      };
      for (int t = blockIdx.x; t < p.total; t += gridDim.x) {
        const auto [b, y0, x0] = conv_tile(t, p.tiles_x, p.tiles_y);
        for (int j = 0; j < 6; ++j) {
          const int s = (int)(u_prep % kNBox);
          if (u_prep >= (uint32_t)kNBox) {
            const uint32_t need = u_prep - (uint32_t)kNBox + 2u;
            while (u_store < need && u_store < u_prep) store_one();
            tma_wait_read<1>();                            // bulk groups retire in order: store #(u_prep - kNBox) has left the box
            if (want_stats || want_shadow) mbar_wait_park(red_done(s), ((u_prep / kNBox) - 1u) & 1u);   // ... and the statistics warp has read it
          }
          c0s[s] = 32 * j; r0s[s] = x0; r1s[s] = y0; r2s[s] = b;
          mbar_expect_tx(in_bar(s), kBoxBytes);
          tma_load_4d(sb + kOffBox + s * kBoxBytes, &tm_x, in_bar(s), 32 * j, x0, y0, b);
          ++u_prep;
        }
      }
      while (u_store < u_prep) store_one();
      tma_wait_all0();
    }
  } else if (warp >= 4) {
    // ===================== compute warps =====================
    const int cw = warp - 4;
    const int cg = cw & 7, rh = cw >> 3;                   // conv role: 8 channels of the slice, output rows 4 rh .. 4 rh + 3 of the tile
    const int gq = lane >> 2, tq = lane & 3;               // MMA fragment coordinates
    const int q = warp & 3, hs = cw >> 2;                  // epilogue role: TMEM lane quarter, 16-column slice of every 64-column group
    const int r = q * 32 + lane;
    const uint32_t rsw = (uint32_t)(r & 7);
    uint8_t* row_ptr = sp + kOffBox + r * 128;
    // per-pixel channel mean / max of a finished tile (the casa gate's 3x3 convs read them, :345-347): the four slice partials of a row
    // are exchanged through s_part2 and flushed by the hs == 0 thread after the NEXT barrier of the compute warps (no extra barrier)
    auto flush_pixel_stats = [&](int tprev, int itprev) {
      if (hs != 0) return;
      const auto [b, y0, x0] = conv_tile(tprev, p.tiles_x, p.tiles_y);
      const int y = y0 + (r >> 4), x = x0 + (r & 15);
      if (y >= p.H || x >= p.W) return;
      const float2* pp = s_part2 + (itprev & 1) * 512;
      float ls = 0.f, lm = -INFINITY;
#pragma unroll
      for (int o = 0; o < 4; ++o) { const float2 tv = pp[o * 128 + r]; ls += tv.x; lm = fmaxf(lm, tv.y); }
      const long long pix = ((long long)b * p.H + y) * p.W + x;
      p.cavg[pix] = ls * (1.0f / (float)kC);
      p.cmax[pix] = lm;
    };
    // ---------- epilogue of one finished tile (iteration index e): x = x + LayerNorm(acc + b2) over the 180 real columns.  It is cut
    // into a statistics pass (epi_begin) and three 64-column groups (epi_group) so that the main loop can interleave it with the conv
    // slices of the NEXT tile: the residual boxes of group g + 1 then have a whole conv slice to be stored, drained and re-loaded, the
    // last fc2 MMA has long retired when its accumulator is read, and the halo load of the next slice hides under epilogue work.
    float e_mean = 0.f, e_rstd = 0.f, e_ls = 0.f, e_lm = -INFINITY;
    auto epi_begin = [&](int e, int tflush) {
      const int as = e & 1;
      mbar_wait(d_full(as), ((uint32_t)(e >> 1)) & 1u);
      tc_fence_after();
      const uint32_t tacc = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * 192);
      // LayerNorm statistics without cancellation: per 16-column group (mean, M2) from registers, merged with Chan's parallel update
      // across the three groups of this thread and then across the four slices of the row
      float n = 0.f, mean = 0.f, m2 = 0.f;
#pragma unroll
      for (int g = 0; g < 3; ++g) {
        const int c0 = 64 * g + 16 * hs;
        float v[16];
        tmem_ld16(tacc + c0, v);
        const int cnt = min(16, max(0, kC - c0));          // 16 except for the last slice of the last group (4 real columns)
        float sg = 0.f, qg = 0.f, mg;
        if (cnt == 16) {
#pragma unroll
          for (int i = 0; i < 16; ++i) { v[i] += s_bias[c0 + i]; sg += v[i]; }
          mg = sg * (1.0f / 16.0f);
#pragma unroll
          for (int i = 0; i < 16; ++i) { const float d = v[i] - mg; qg = fmaf(d, d, qg); }
        } else {
#pragma unroll
          for (int i = 0; i < 16; ++i) { v[i] += s_bias[c0 + i]; if (i < cnt) sg += v[i]; }
          mg = sg / (float)max(cnt, 1);
#pragma unroll
          for (int i = 0; i < 16; ++i) { const float d = v[i] - mg; if (i < cnt) qg = fmaf(d, d, qg); }
        }
        if (cnt > 0) {
          const float nn = n + (float)cnt, d = mg - mean;
          mean += d * ((float)cnt / nn);
          m2 += qg + d * d * (n * (float)cnt / nn);
          n = nn;
        }
      }
      float2* part = s_part + (e & 1) * 512;
      part[hs * 128 + r] = make_float2(mean, m2);
      named_bar_sync(q + 1, 128);   // the four compute warps that share TMEM lane quarter q exchange their partials
      if (want_stats && tflush >= 0) flush_pixel_stats(tflush, e - 1);
#pragma unroll
      for (int o = 1; o < 4; ++o) {
        const int ho = (hs + o) & 3;
        const float2 tv = part[ho * 128 + r];
        const float cnt = ho == 3 ? 36.f : 48.f;           // real columns of slice ho: 3 x 16, the last slice ends at column 180
        const float nn = n + cnt, d = tv.x - mean;
        mean += d * (cnt / nn);
        m2 += tv.y + d * d * (n * cnt / nn);
        n = nn;
      }
      e_mean = mean;
      e_rstd = rsqrtf(m2 * (1.0f / (float)kC) + 1e-5f);
      e_ls = 0.f; e_lm = -INFINITY;                         // channel sum / max of this thread's real output columns
    };
    auto epi_group = [&](int e, int g) {
      const int as = e & 1;
      const uint32_t tacc = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * 192);
      const int c0 = 64 * g + 16 * hs;
      float v[16];
      tmem_ld16(tacc + c0, v);
#pragma unroll
      for (int i = 0; i < 16; ++i) v[i] = fmaf((v[i] + s_bias[c0 + i] - e_mean) * e_rstd, s_gamma[c0 + i], s_beta[c0 + i]);   // gamma = beta = 0 beyond 180
      const uint32_t ub = (uint32_t)e * 6u + (uint32_t)(2 * g + (hs >> 1));
      const int bb = (int)(ub % kNBox);
      mbar_wait(in_bar(bb), (ub / kNBox) & 1u);
      uint8_t* fb = row_ptr + bb * kBoxBytes;
      const uint32_t ch0 = (uint32_t)((hs & 1) * 4);
#pragma unroll
      for (int ch = 0; ch < 4; ++ch) {
        float4* ptr = reinterpret_cast<float4*>(fb + (((ch0 + (uint32_t)ch) ^ rsw) << 4));
        const float4 rr = *ptr;
        const float4 o = make_float4(v[4 * ch] + rr.x, v[4 * ch + 1] + rr.y, v[4 * ch + 2] + rr.z, v[4 * ch + 3] + rr.w);
        *ptr = o;
        if (c0 + 4 * ch < kC) {                             // 180 = 45 chunks of 4: a chunk is entirely real or entirely padding
          e_ls += (o.x + o.y) + (o.z + o.w);
          e_lm = fmaxf(e_lm, fmaxf(fmaxf(o.x, o.y), fmaxf(o.z, o.w)));
        }
      }
      fence_proxy_async_smem();
      mbar_arrive_warp(out_bar(bb));
      if (g == 2) {
        tc_fence_before();
        mbar_arrive_warp(d_empty(as));
        if (want_stats) s_part2[(e & 1) * 512 + hs * 128 + r] = make_float2(e_ls, e_lm);   // flushed after the next tile's LayerNorm barrier
      }
    };
    // ldmatrix row of this lane: matrix m = lane >> 3 holds pixels (m & 1) * 8 .. + 7 of tap dx + (m >> 1); four byte offsets cover the
    // swizzle classes (pixel & 7) that the even window origins 4 yi + 2 s can take (the halo row pitch is 20 = 4 mod 8 pixels)
    const uint32_t lj = (uint32_t)((lane & 7) + ((lane >> 3) & 1) * 8 + (lane >> 4));
    uint32_t swz[4];
#pragma unroll
    for (int c4 = 0; c4 < 4; ++c4)
      swz[c4] = sb + kOffHalo + (uint32_t)(rh * 4 * kPW) * 128u + lj * 128u + ((((uint32_t)cg) ^ ((lj + 2u * (uint32_t)c4) & 7u)) << 4);
    // fc2 A-operand word of this lane: tile pixel row (4 rh + yo) * 16 + gq (+ 8), 16-byte chunk cg, channel pair tq
    const uint32_t a_off = (uint32_t)(rh * 4 * 16 + gq) * 128u + ((((uint32_t)cg) ^ (uint32_t)gq) << 4) + (uint32_t)tq * 4u;
    int it = 0, tprev = -1, tpp = -1;
    for (int t = blockIdx.x; t < p.total; t += gridDim.x, ++it) {
      // ---------- depthwise 5x5 + GELU + input, slice by slice -> A operand; after every second slice one group of the previous tile's epilogue.
      // One m16n8k16 MMA covers 16 pixels of an image row (M), 8 channels (N) and two horizontal taps (K = tap x channel, B = diag(w_tap)
      // blocks), so an output row takes 13 MMAs (10 for taps dx = 0..3, 3 for the dx = 4 column paired vertically).  A fragments come from ldmatrix (a matrix row = 8 channels of one pixel = one 16-byte
      // chunk): the SWIZZLE_128B halo box puts the 8 pixels of a matrix on 8 different bank groups, so every load is conflict-free.
#pragma unroll 1
      for (int k = 0; k < 6; ++k) {
        const int h = k & 1;
        const uint32_t u = (uint32_t)(it * 3 + (k >> 1));
        // tap rows [64 channels][28 words]: 5 x (taps dx = 0..3 of row ky), then (0,4) (1,4) (2,4) (3,4), then (4,4) 0 bias 0 -- the order in which
        // the MMAs pair them.  B[k = channel][n = channel] is diagonal: only the lane with tq == gq / 2 holds non-zero words (in the half chosen
        // by the channel parity at pack time); every other lane reads the zero row, so the whole set-up is seven 16-byte loads.
        const uint32_t* tblu = reinterpret_cast<const uint32_t*>(sp + kOffHalo + h * kHaloStage + kHalo);
        uint8_t* abuf = sp + kOffA + h * kABuf;
        const uint32_t hoff = (uint32_t)(h * kHaloStage);
        mbar_wait(halo_full(h), u & 1u);
        const uint4* brow = (tq == (gq >> 1)) ? reinterpret_cast<const uint4*>(tblu + (cg * 8 + gq) * kDwRow) : reinterpret_cast<const uint4*>(sp + kOffZero);
        uint4 bq[7];
#pragma unroll
        for (int i = 0; i < 7; ++i) bq[i] = brow[i];
        const float2 bs = make_float2(__uint_as_float(tblu[(cg * 8 + 2 * tq) * kDwRow + 26]), __uint_as_float(tblu[(cg * 8 + 2 * tq + 1) * kDwRow + 26]));
        const bool live = k * 64 + cg * 8 + 2 * tq < kHid;
        float acc[4][4];
#pragma unroll
        for (int y = 0; y < 4; ++y) { acc[y][0] = bs.x; acc[y][1] = bs.y; acc[y][2] = bs.x; acc[y][3] = bs.y; }
        uint32_t cen[4][2];
        uint32_t P4[2] = {0u, 0u};                                                         // dx = 4 fragments of the previous input row
#pragma unroll
        for (int yr = 0; yr < 8; ++yr) {                                                   // input row 4 rh + yr of the halo box
          uint32_t F[5][2];
#pragma unroll
          for (int sx = 0; sx < 2; ++sx)
            ldmatrix_x4(swz[((4 * yr + 2 * sx) & 7) >> 1] + hoff + (uint32_t)((yr * kPW + 2 * sx) * 128), F[2 * sx][0], F[2 * sx][1], F[2 * sx + 1][0], F[2 * sx + 1][1]);
          ldmatrix_x2(swz[((4 * yr + 4) & 7) >> 1] + hoff + (uint32_t)((yr * kPW + 4) * 128), F[4][0], F[4][1]);
          if (yr == 7) mbar_arrive_warp(halo_empty(h));                                    // every input word of this warp is in registers
#pragma unroll
          for (int sx = 0; sx < 2; ++sx)                                                   // taps dx = 0..3 in pairs; consecutive MMAs go to different output rows
#pragma unroll
            for (int ky = 0; ky < 5; ++ky) {
              const int yo = yr - ky;                                                      // compile-time after unrolling
              if (yo >= 0 && yo < 4) mma_bf16_16816(acc[yo], F[2 * sx][0], F[2 * sx][1], F[2 * sx + 1][0], F[2 * sx + 1][1], sx ? bq[ky].z : bq[ky].x, sx ? bq[ky].w : bq[ky].y);
            }
          // the dx = 4 column pairs vertically: taps (0,4)+(1,4) and (2,4)+(3,4) take this row and the previous one, (4,4) stays single
          if (yr - 1 >= 0 && yr - 1 < 4) mma_bf16_16816(acc[yr - 1], P4[0], P4[1], F[4][0], F[4][1], bq[5].x, bq[5].y);
          if (yr - 3 >= 0 && yr - 3 < 4) mma_bf16_16816(acc[yr - 3], P4[0], P4[1], F[4][0], F[4][1], bq[5].z, bq[5].w);
          if (yr - 4 >= 0 && yr - 4 < 4) mma_bf16_16816(acc[yr - 4], F[4][0], F[4][1], 0u, 0u, bq[6].x, bq[6].y);
          P4[0] = F[4][0]; P4[1] = F[4][1];
          if (yr >= 2 && yr < 6) { cen[yr - 2][0] = F[2][0]; cen[yr - 2][1] = F[2][1]; }
        }
        // GELU + input -> fc2 A operand for all 8 channel pairs of this lane at once: eight independent ex2 / rcp chains hide the MUFU latency
        mbar_wait(a_empty(h), (u & 1u) ^ 1u);                                              // the fc2 MMAs of the previous use of this A buffer are done
#pragma unroll
        for (int yo = 0; yo < 4; ++yo)
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
            const float2 cv = unpack_bf16x2_alu(cen[yo][hh]);
            const float2 gl = gelu2(make_float2(acc[yo][2 * hh], acc[yo][2 * hh + 1]));
            const float2 h2 = __fadd2_rn(cv, gl);
            const uint32_t o = live ? pack_bf16x2(h2.x, h2.y) : 0u;
            *reinterpret_cast<uint32_t*>(abuf + (yo * 16 + 8 * hh) * 128 + a_off) = o;
          }
        fence_proxy_async_smem();
        mbar_arrive_warp(a_full(h));
        if (it > 0 && h == 1) {
          if (k == 1) epi_begin(it - 1, tpp);
          epi_group(it - 1, k >> 1);
        }
      }
      tpp = tprev; tprev = t;
    }
    if (it > 0) {                                           // the last tile's epilogue has nothing to hide behind
      epi_begin(it - 1, tpp);
      for (int g = 0; g < 3; ++g) epi_group(it - 1, g);
    }
    if (want_stats && tprev >= 0) { named_bar_sync(q + 1, 128); flush_pixel_stats(tprev, it - 1); }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace

// h1: bf16 [B,H,W,384]; dw_tbl_mma: depthwise tap rows (launch_pack_dw_mma); w2_img: fc2 operand images (launch_pack_w2_image);
// x: fp32 residual stream [B,H,W,180], updated in place
int launch_ffn_tail(const bf16* h1, const uint32_t* dw_tbl_mma, const uint8_t* w2_img, const float* b2, const float* gamma,
                    const float* beta, float* x, int B, int H, int W, const FfnStats* stats, bf16* shadow, int num_sms, cudaStream_t st,
                    const FfnBand* band) {
  static unsigned long long configured = 0;
  if (ensure_dynamic_smem(ffn_tail_kernel, kSmemBytes, &configured)) return 1;
  Params p;
  p.B = B; p.H = H; p.W = W;
  p.tiles_x = cdiv(W, kConvTileW); p.tiles_y = cdiv(H, kConvTileH);
  const long long total = (long long)B * p.tiles_x * p.tiles_y;
  if (total > 2147483647LL / 8) { set_error("launch_ffn_tail: too many tiles"); return 1; }
  p.total = (int)total;
  p.bias = b2; p.gamma = gamma; p.beta = beta;
  p.cavg = p.cmax = p.part_sum = p.part_max = nullptr; p.Hp = H; p.Wp = W;
  p.shadow = stats == nullptr ? shadow : nullptr;          // the statistics warp does one or the other
  if (stats != nullptr) { p.cavg = stats->cavg; p.cmax = stats->cmax; p.part_sum = stats->part_sum; p.part_max = stats->part_max; p.Hp = stats->Hp; p.Wp = stats->Wp; }
  p.dw_tbl = dw_tbl_mma; p.w2_img = w2_img;
  p.h1_y_off = band ? band->halo : 0; p.yg0 = band ? band->yg0 : 0; p.Hf = band ? band->Hf : H;
  if (band && B != 1) { set_error("launch_ffn_tail: band mode needs B == 1"); return 1; }
  CUtensorMap tm_h1, tm_x;
  // SWIZZLE_128B halo boxes, zero fill outside the image; band mode: the map starts h1_y_off rows above image row 0 (rows filled by the neighbour)
  if (make_tmap_nhwc(&tm_h1, h1 - (size_t)p.h1_y_off * W * kHidp, B, H + 2 * p.h1_y_off, W, kHidp, 64, kPW, kPH)) return 1;
  if (make_tmap_nhwc_t(&tm_x, x, 4, B, H, W, kC, kC, 32, 16, 8)) return 1;
  const int grid = p.total < num_sms ? p.total : num_sms;
  HITSIR_CHECK(launch_pdl(ffn_tail_kernel, dim3(grid), dim3(640), kSmemBytes, st, tm_h1, tm_x, p));
  return 0;
}

}  // namespace hitsir
