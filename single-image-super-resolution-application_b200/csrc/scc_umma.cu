// Spatial-channel self-correlation inside hierarchical windows on tcgen05 tensor cores
// (SCC.forward without the final proj, /root/reference/models/hit_sir_pro.py:542-596).
//
// Reference math per window (L = w*w tokens, pooled grid of Lb = min(w,8)^2 cells, r = w/min(w,8)):
//   token t = [q | v] (2 x 6 heads x 15)                                             (:569-570)
//   k  = (Wk1 q_h + bk1 + Wk2 v_h + bk2) / 2  per head, weights shared by the heads   (:572)
//   kp = pool(k), vp = pool(v): cell = sum_{i,j<r} wsl[i*r+j] * tok + bsl             (:451-455)
//   S-SC: out_s[l,h,:] = sum_m (q_lh . kp[m,h] / 15 + bias[h,l,m]) * vp[m,h,:]        (:475,503,511)
//   C-SC: corr[c,c'] = sum_l q[l,c] k[l,c'] / L ;  out_c[l,c] = sum_c' corr[c,c'] v[l,c']   (:531,538)
//
// B200 formulation.  No softmax anywhere, so everything is linear algebra that can be re-associated
// into dense contractions over *raw* tokens (k-gen and pooling commute with the window reductions):
//   phase A (reduce over the window's tokens, operands straight from the TMA-loaded token tile):
//       G   = Q^T T            [96 x 192]   (token tile as MN-major A and B operands, K = tokens)
//       TPT = T^T Pool^T       [192 x 64]   (pooled raw tokens, transposed; Pool = weights-only image)
//   mid (per window, five tiny steps alternating tensor core <-> epilogue warps):
//       corr = G  Wk^T / L     KP = TPT^T Wk^T + bsl      VPT = TPT[v rows] + bsl
//       Mh   = KP_h^T VP_h / 15  (6 diagonal 16x16 blocks)
//   phase B (per 128-token tile, one accumulator [128 x 192]):
//       out_s = Q Mblk + sum_h Bias_h[128 x 64] VP_h       out_c = V corr^T
// The token layout is head-padded (6 x 16 | 6 x 16 = 192 channels, kernels.cuh scc_pos); position 15 holds a
// constant 1 so that the k-gen bias rides along in the contractions.
//
// Serves the windows with pooling ratio r > 1: w = 16, 32, 48, 64 (two or more 128-token tiles of 16x8 pixels), and w = 4 / 8 when
// base_win_size is below the window (one tile: resident mode).  Windows with r = 1 run in scc_dense.cu.
// One persistent CTA per SM walks whole windows.  Warp roles: warp 0 = TMA producer, warp 1 = MMA issuer,
// warp 2 = TMEM allocator, warp 3 = TMA-store thread, warps 4..11 = TMEM->register->smem converters / epilogue.
#include "gemm.cuh"
#include "kernels.cuh"

namespace hitsir {

namespace {

constexpr int kBlk = 16384;                 // one 64-channel block of a token tile: 128 rows x 128 B
constexpr int kStage = 3 * kBlk;            // token tile stage
constexpr int kSlot = 16384;                // ring slot (pool chunk / one head's bias chunk)
constexpr int kSlots = 4;
constexpr int kGBlk = 96 * 128;             // block stride of the 96-row operand images (G, corr)
constexpr int kOffRing = 2 * kStage;
constexpr int kOffG = kOffRing;                       // bf16 G  [96][192]   (ring slots 0..2 between phase A and mid2)
constexpr int kOffKP = kOffRing + 3 * kSlot;          // ring slot 3: raw pooled v rows [96][64] (mid1..mid2), then bf16 KP [64][96] as 2 blocks of 8 KB (mid3..mid4)
constexpr int kOffTPT = kOffRing + kSlots * kSlot;    // bf16 TPT [192][64]; rows 96.. are VPT (live through phase B)
constexpr int kOffCorr = kOffTPT + 192 * 128;         // bf16 corr [96][2 blocks]
constexpr int kOffMblk = kOffCorr + 2 * kGBlk;        // bf16 Mblk [96][128 B]
constexpr int kOffW = kOffMblk + kGBlk;               // k-gen operand image [16][128 B]
constexpr int kOffBars = kOffW + 2048;
constexpr int kNumBars = 25;
// resident mode (one tile per window): stage s keeps its compact token blocks in the first 24 KB of its 48 KB region, head h's bias
// image sits at kResBias(h); the pool image follows the three G blocks
constexpr int kOffResPool = kOffG + 3 * kGBlk;
__host__ __device__ constexpr int res_bias_off(int h, int bias_bytes) { return (h / 3) * kStage + 24576 + (h % 3) * bias_bytes; }
constexpr int kSmemBytes = kOffBars + kNumBars * 8 + 16 + 1024;
static_assert(kSmemBytes <= 232448, "smem budget");

// TMEM columns
constexpr int kTmG = 0, kTmTlo = 192, kTmThi = 256, kTmCorr = 320, kTmKP = 416, kTmMblk = 320;

struct Params {
  int nwin, nWx, nWy;
  int w, bx, by, TT, tiles_x, tiles, ksteps;
  int Lb, streaming;
  int cell_ksteps;           // ceil(Lb / 16): k-steps of the contractions over pooled cells
  int resident;              // single-tile windows (w = 4, 8): pool / bias operand images stay in shared memory, tokens are prefetched
  int blk;                   // byte stride between the three 64-channel blocks of a token stage (kBlk, or TT*128 when resident)
  float invL;
  int pool_bytes, bias_bytes;
  const uint8_t* pool_img;   // [tiles][pool_bytes]
  const uint8_t* bias_img;   // [tiles][6][bias_bytes]
  const uint8_t* w_img;      // 2 KB
  const float* bsl;          // spatial_linear.bias (device scalar)
  int H, W;                  // unpadded image size (stores outside are skipped / clipped)
};

__global__ void __launch_bounds__(384, 1)
scc_umma_kernel(const __grid_constant__ CUtensorMap tm_t, const __grid_constant__ CUtensorMap tm_o, const Params p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sb = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sp = smem_raw + (sb - smem_u32(smem_raw));
  const uint32_t bar0 = sb + kOffBars;
  auto tok_full = [&](int s) { return bar0 + 8u * s; };
  auto tok_empty = [&](int s) { return bar0 + 8u * (2 + s); };
  auto ring_full = [&](int s) { return bar0 + 8u * (4 + s); };
  auto ring_empty = [&](int s) { return bar0 + 8u * (8 + s); };
  const uint32_t a_done = bar0 + 8u * 12, mid1_done = bar0 + 8u * 13, mid2_ready = bar0 + 8u * 14, mid3_done = bar0 + 8u * 15,
                 mid4_ready = bar0 + 8u * 16, mid5_done = bar0 + 8u * 17;
  auto d_full = [&](int s) { return bar0 + 8u * (18 + s); };
  auto d_empty = [&](int s) { return bar0 + 8u * (20 + s); };
  auto st_ready = [&](int s) { return bar0 + 8u * (22 + s); };
  const uint32_t res_full = bar0 + 8u * 24;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(sp + kOffBars + kNumBars * 8);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) { tma_prefetch_desc(&tm_t); tma_prefetch_desc(&tm_o); }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < 2; ++s) { mbar_init(tok_full(s), 1); mbar_init(tok_empty(s), 1); }
    for (int s = 0; s < kSlots; ++s) { mbar_init(ring_full(s), 1); mbar_init(ring_empty(s), 1); }
    mbar_init(a_done, 1); mbar_init(mid1_done, 8); mbar_init(mid2_ready, 1); mbar_init(mid3_done, 8);
    mbar_init(mid4_ready, 1); mbar_init(mid5_done, 8);
    mbar_init(res_full, 1);
    for (int s = 0; s < 2; ++s) { mbar_init(d_full(s), 1); mbar_init(d_empty(s), 8); mbar_init(st_ready(s), 8); }
    fence_barrier_init();
  }
  if (warp == 2) { tmem_alloc(smem_u32(tmem_ptr_smem), 512); tmem_relinquish(); }
  for (int i = threadIdx.x; i < 2048 / 16; i += blockDim.x)
    reinterpret_cast<uint4*>(sp + kOffW)[i] = reinterpret_cast<const uint4*>(p.w_img)[i];
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_ptr_smem;
  const int mult = p.streaming ? 2 : 1;
  pdl_entry();                                           // up to here only the weights-only k-gen image was read

  if (warp == 0) {
    if (lane == 0) {
      // ===================== producer =====================
      uint32_t tok_cnt = 0, ring_cnt = 0;
      int wi = 0;
      auto load_tokens = [&](int b, int x0, int y0) {
        const int s = (int)(tok_cnt & 1u);
        wait_bar(tok_empty(s), ((tok_cnt >> 1) & 1u) ^ 1u);
        mbar_expect_tx(tok_full(s), (uint32_t)(p.TT * 128 * 3));
#pragma unroll
        for (int blk = 0; blk < 3; ++blk) tma_load_4d(sb + s * kStage + blk * p.blk, &tm_t, tok_full(s), blk * 64, x0, y0, b);
        ++tok_cnt;
      };
      auto load_chunk = [&](const uint8_t* src, uint32_t bytes) {
        const int r = (int)(ring_cnt & 3u);
        wait_bar(ring_empty(r), ((ring_cnt >> 2) & 1u) ^ 1u);
        mbar_expect_tx(ring_full(r), bytes);
        bulk_load(sb + kOffRing + r * kSlot, src, bytes, ring_full(r));
        ++ring_cnt;
      };
      if (p.resident) {
        mbar_expect_tx(res_full, (uint32_t)(p.pool_bytes + kHeads * p.bias_bytes));
        bulk_load(sb + kOffResPool, p.pool_img, (uint32_t)p.pool_bytes, res_full);
        for (int h = 0; h < kHeads; ++h)
          bulk_load(sb + res_bias_off(h, p.bias_bytes), p.bias_img + (size_t)h * p.bias_bytes, (uint32_t)p.bias_bytes, res_full);
        for (int win = blockIdx.x; win < p.nwin; win += gridDim.x) {
          const int wx = win % p.nWx; const int t2 = win / p.nWx; const int wy = t2 % p.nWy; const int b = t2 / p.nWy;
          load_tokens(b, wx * p.w, wy * p.w);          // runs ahead by one window (two stages)
        }
      } else
      for (int win = blockIdx.x; win < p.nwin; win += gridDim.x, ++wi) {
        const int wx = win % p.nWx; const int t2 = win / p.nWx; const int wy = t2 % p.nWy; const int b = t2 / p.nWy;
        for (int t = 0; t < p.tiles; ++t) {
          const int x0 = wx * p.w + (t % p.tiles_x) * p.bx, y0 = wy * p.w + (t / p.tiles_x) * p.by;
          load_tokens(b, x0, y0);
          load_chunk(p.pool_img + (size_t)t * p.pool_bytes, (uint32_t)p.pool_bytes);
        }
        wait_bar(mid4_ready, (uint32_t)(wi & 1));      // ring slots double as G / KP operand storage until then
        for (int tb = 0; tb < p.tiles; ++tb) {
          // streamed windows walk phase B backwards: the tiles phase A read last are the ones most likely to be in L2 still (148 CTAs x
          // 18-32 tiles x 48 KB is more than the 126 MB L2, re-reading in the same order missed on every tile)
          const int t = p.streaming ? p.tiles - 1 - tb : tb;
          if (p.streaming) {
            const int x0 = wx * p.w + (t % p.tiles_x) * p.bx, y0 = wy * p.w + (t / p.tiles_x) * p.by;
            load_tokens(b, x0, y0);
          }
          for (int h = 0; h < kHeads; ++h) load_chunk(p.bias_img + ((size_t)t * kHeads + h) * p.bias_bytes, (uint32_t)p.bias_bytes);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ===================== MMA issuer =====================
      constexpr uint32_t id_G = make_idesc(128, 192, 1, 1);      // Q^T T : both operands MN-major views of the token tile
      constexpr uint32_t id_T = make_idesc(128, 64, 1, 0);       // T^T Pool^T
      constexpr uint32_t id_c16 = make_idesc(128, 16, 0, 0);     // G_h Wk^T, Q_h Mh, Bias_h VP_h
      constexpr uint32_t id_kp = make_idesc(128, 16, 1, 0);      // TPT^T Wk^T
      constexpr uint32_t id_mb = make_idesc(128, 96, 0, 1);      // VPT KP
      constexpr uint32_t id_oc = make_idesc(128, 96, 0, 0);      // V corr^T
      uint32_t tok_cnt = 0, ring_cnt = 0, d_cnt = 0;
      int wi = 0;
      if (p.resident) wait_bar(res_full, 0u);
      for (int win = blockIdx.x; win < p.nwin; win += gridDim.x, ++wi) {
        // the phase-A accumulators overlay both phase-B buffers of the previous window
        for (uint32_t buf = 0; buf < 2; ++buf)
          if (d_cnt > buf) { const uint32_t last = ((d_cnt - 1 - buf) >> 1 << 1) + buf; wait_bar(d_empty((int)buf), (last >> 1) & 1u); }
        tc_fence_after();
        const uint32_t a0 = tok_cnt;
        // ---------- phase A
        for (int t = 0; t < p.tiles; ++t) {
          const int s = (int)(tok_cnt & 1u);
          wait_bar(tok_full(s), (tok_cnt >> 1) & 1u);
          const int r = (int)(ring_cnt & 3u);
          if (!p.resident) wait_bar(ring_full(r), (ring_cnt >> 2) & 1u);
          tc_fence_after();
          const uint32_t st = sb + s * kStage, pool = p.resident ? sb + kOffResPool : sb + kOffRing + r * kSlot;
          for (int ks = 0; ks < p.ksteps; ++ks) {
            const uint32_t acc = (t | ks) != 0 ? 1u : 0u;
            const uint64_t da = make_desc(st + ks * 2048, (uint32_t)p.blk, 1024);
            const uint64_t da2 = make_desc(st + 2 * p.blk + ks * 2048, (uint32_t)p.blk, 1024);
            const uint64_t dp = umma_desc_sw128(pool + (ks >> 2) * 8192 + (ks & 3) * 32);
            umma_bf16(tmem + kTmG, da, da, id_G, acc);
            umma_bf16(tmem + kTmTlo, da, dp, id_T, acc);
            umma_bf16(tmem + kTmThi, da2, dp, id_T, acc);
          }
          if (!p.resident) { umma_commit(ring_empty(r)); ++ring_cnt; }
          if (p.streaming) umma_commit(tok_empty(s));
          ++tok_cnt;
        }
        umma_commit(a_done);
        // ---------- mid2: corr = G Wk^T, KP = TPT^T Wk^T (per head: q part, v part, bias via the ones channel)
        wait_bar(mid1_done, (uint32_t)(wi & 1));
        tc_fence_after();
        {
          // every head's q slice carries its own ones column (position 16h+15), so the k-gen bias rides in the q-part contraction.
          // Issue order interleaves the 12 independent accumulators: back-to-back MMAs never accumulate into the same columns.
          const uint32_t gb = sb + kOffG, tb = sb + kOffTPT, wb = sb + kOffW;
          const uint64_t w1d = umma_desc_sw128(wb), w2d = umma_desc_sw128(wb + 32);
#pragma unroll
          for (int h = 0; h < kHeads; ++h) {
            umma_bf16(tmem + kTmCorr + 16 * h, umma_desc_sw128(gb + (h >> 2) * kGBlk + (h & 3) * 32), w1d, id_c16, 0u);
            umma_bf16(tmem + kTmKP + 16 * h, make_desc(tb + 16 * h * 128, 1024, 1024), w1d, id_kp, 0u);
          }
#pragma unroll
          for (int h = 0; h < kHeads; ++h) {
            const int cv = 96 + 16 * h;
            umma_bf16(tmem + kTmCorr + 16 * h, umma_desc_sw128(gb + (cv >> 6) * kGBlk + (cv & 63) * 2), w2d, id_c16, 1u);
            umma_bf16(tmem + kTmKP + 16 * h, make_desc(sb + kOffKP + 16 * h * 128, 1024, 1024), w2d, id_kp, 1u);
          }
        }
        umma_commit(mid2_ready);
        // ---------- mid4: Mfull[(h,j)][(h',i)] = sum_m VPT[(h,j)][m] KP[m][(h',i)]
        wait_bar(mid3_done, (uint32_t)(wi & 1));
        tc_fence_after();
        for (int ks = 0; ks < p.cell_ksteps; ++ks)
          umma_bf16(tmem + kTmMblk, umma_desc_sw128(sb + kOffTPT + 96 * 128 + ks * 32), make_desc(sb + kOffKP + ks * 2048, 8192, 1024), id_mb, ks ? 1u : 0u);
        umma_commit(mid4_ready);
        // ---------- phase B
        wait_bar(mid5_done, (uint32_t)(wi & 1));
        tc_fence_after();
        for (int t = 0; t < p.tiles; ++t) {
          const uint32_t idx = p.streaming ? tok_cnt : a0 + (uint32_t)t;
          const int s = (int)(idx & 1u);
          if (p.streaming) { wait_bar(tok_full(s), (idx >> 1) & 1u); ++tok_cnt; }
          const int buf = (int)(d_cnt & 1u);
          wait_bar(d_empty(buf), ((d_cnt >> 1) & 1u) ^ 1u);
          tc_fence_after();
          const uint32_t st = sb + s * kStage, D = tmem + (uint32_t)(buf * 192);
          auto corr_step = [&](int ks) {
            const int ch = 96 + 16 * ks;
            umma_bf16(D + 96, umma_desc_sw128(st + (ch >> 6) * p.blk + (ch & 63) * 2), umma_desc_sw128(sb + kOffCorr + ((ch >> 6) - 1) * kGBlk + (ch & 63) * 2), id_oc,
                      ks ? 1u : 0u);
          };
          if (p.resident) {
            // all six bias images are resident: interleave the seven independent accumulators (6 heads + out_c)
#pragma unroll
            for (int h = 0; h < kHeads; ++h)
              umma_bf16(D + 16 * h, umma_desc_sw128(st + (h >> 2) * p.blk + (h & 3) * 32), umma_desc_sw128(sb + kOffMblk + 16 * h * 128 + (h & 3) * 32), id_c16, 0u);
            corr_step(0);
            for (int ks = 0; ks < p.cell_ksteps; ++ks) {
#pragma unroll
              for (int h = 0; h < kHeads; ++h)
                umma_bf16(D + 16 * h, umma_desc_sw128(sb + res_bias_off(h, p.bias_bytes) + ks * 32), umma_desc_sw128(sb + kOffTPT + (96 + 16 * h) * 128 + ks * 32), id_c16, 1u);
              if (ks + 1 < 6) corr_step(ks + 1);
            }
            for (int ks = p.cell_ksteps + 1; ks < 6; ++ks) corr_step(ks);
          } else {
            for (int h = 0; h < kHeads; ++h) {
              umma_bf16(D + 16 * h, umma_desc_sw128(st + (h >> 2) * p.blk + (h & 3) * 32), umma_desc_sw128(sb + kOffMblk + 16 * h * 128 + (h & 3) * 32), id_c16, 0u);
              corr_step(h);
              const int r = (int)(ring_cnt & 3u);
              wait_bar(ring_full(r), (ring_cnt >> 2) & 1u);
              tc_fence_after();
              const uint32_t bias = sb + kOffRing + r * kSlot, vp = sb + kOffTPT + (96 + 16 * h) * 128;
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) umma_bf16(D + 16 * h, umma_desc_sw128(bias + ks * 32), umma_desc_sw128(vp + ks * 32), id_c16, 1u);
              umma_commit(ring_empty(r));
              ++ring_cnt;
            }
          }
          umma_commit(d_full(buf));
          ++d_cnt;
        }
      }
    }
  } else if (warp == 3) {
    if (lane == 0) {
      // ===================== TMA store of finished tiles =====================
      uint32_t tok_cnt = 0, st_cnt[2] = {0, 0};
      for (int win = blockIdx.x; win < p.nwin; win += gridDim.x) {
        const int wx = win % p.nWx; const int t2 = win / p.nWx; const int wy = t2 % p.nWy; const int b = t2 / p.nWy;
        const uint32_t a0 = tok_cnt;
        for (int tb = 0; tb < p.tiles; ++tb) {
          const uint32_t idx = p.streaming ? a0 + (uint32_t)(p.tiles + tb) : a0 + (uint32_t)tb;
          const int s = (int)(idx & 1u);
          wait_bar(st_ready(s), st_cnt[s] & 1u);
          ++st_cnt[s];
          const int t = p.streaming ? p.tiles - 1 - tb : tb;      // phase-B order of the producer
          const int x0 = wx * p.w + (t % p.tiles_x) * p.bx, y0 = wy * p.w + (t / p.tiles_x) * p.by;
          if (x0 < p.W && y0 < p.H) {                 // tiles entirely inside the reflect padding are cropped (:696)
#pragma unroll
            for (int blk = 0; blk < 3; ++blk) tma_store_4d(&tm_o, sb + s * kStage + blk * p.blk, blk * 64, x0, y0, b);
            tma_commit();
            tma_wait_read<0>();
          }
          mbar_arrive(tok_empty(s));
        }
        tok_cnt = a0 + (uint32_t)(mult * p.tiles);
      }
      tma_wait_all0();
    }
  } else if (warp >= 4) {
    // ===================== converters / epilogue (8 warps) =====================
    const int q = warp & 3, hs = (warp - 4) >> 2;
    const int row = q * 32 + lane;
    const uint32_t tl = tmem + ((uint32_t)(q * 32) << 16);
    const float bsl = *p.bsl;
    uint32_t tok_cnt = 0, d_cnt = 0;
    int wi = 0;
    for (int win = blockIdx.x; win < p.nwin; win += gridDim.x, ++wi) {
      const uint32_t par = (uint32_t)(wi & 1);
      // ---------- mid1: G, TPT -> bf16 operand images
      wait_bar(a_done, par);
      tc_fence_after();
      if (q < 3) {
        float v[6][16];
        tmem_ld_cols<6>(tl + kTmG + hs * 96, v);
#pragma unroll
        for (int i = 0; i < 6; ++i) {
          const int c0 = hs * 96 + 16 * i;
          store16(sp + kOffG + (c0 >> 6) * kGBlk, row, (c0 & 63) >> 3, v[i]);
        }
      }
      if (hs == 0 || q < 2) {
        const int crow = hs == 0 ? row : 128 + row;
        const uint32_t src = tl + (hs == 0 ? kTmTlo : kTmThi);
        const bool vrow = crow >= 96;
        const bool padrow = ((crow - 96) & 15) == 15;
        float v[4][16];
        tmem_ld_cols<4>(src, v);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          if (vrow) {
            // raw pooled v rows feed the k-gen contraction (KP) from ring slot 3; the TPT image keeps vp = pooled v + bsl
            store16(sp + kOffKP, crow - 96, 2 * i, v[i]);
#pragma unroll
            for (int e = 0; e < 16; ++e) v[i][e] = (16 * i + e < p.Lb && !padrow) ? v[i][e] + bsl : 0.f;
          }
          store16(sp + kOffTPT, crow, 2 * i, v[i]);
        }
      }
      tc_fence_before();
      fence_proxy_async_smem();
      mbar_arrive_warp(mid1_done);
      // ---------- mid3: corr, KP -> bf16 operand images
      wait_bar(mid2_ready, par);
      tc_fence_after();
      if (q < 3) {
        float v[3][16];
        tmem_ld_cols<3>(tl + kTmCorr + hs * 48, v);
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          const int c0 = hs * 48 + 16 * i, ch = 96 + c0;
#pragma unroll
          for (int e = 0; e < 16; ++e) v[i][e] *= p.invL;
          store16(sp + kOffCorr + ((ch >> 6) - 1) * kGBlk, row, (ch & 63) >> 3, v[i]);
        }
      }
      if (q < 2) {
        float v[3][16];
        tmem_ld_cols<3>(tl + kTmKP + hs * 48, v);
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          const int c0 = hs * 48 + 16 * i;
#pragma unroll
          for (int e = 0; e < 16; ++e) v[i][e] = (row < p.Lb && e != 15) ? v[i][e] + bsl : 0.f;
          store16(sp + kOffKP + (c0 >> 6) * 8192, row, (c0 & 63) >> 3, v[i]);
        }
      }
      tc_fence_before();
      fence_proxy_async_smem();
      mbar_arrive_warp(mid3_done);
      // ---------- mid5: diagonal blocks of Mfull / 15 -> Mblk operand image
      wait_bar(mid4_ready, par);
      tc_fence_after();
      if (hs == 0 && q < 3) {
        float v[2][16];
        tmem_ld_cols<2>(tl + kTmMblk + 32 * q, v);
        const int h = row >> 4;
        float o[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) o[e] = ((lane & 16) ? v[1][e] : v[0][e]) * (1.0f / 15.0f);
        store16(sp + kOffMblk, row, 2 * (h & 3), o);
      }
      tc_fence_before();
      fence_proxy_async_smem();
      mbar_arrive_warp(mid5_done);
      // ---------- phase B epilogue: accumulator -> bf16, in place over the consumed token tile, then TMA store
      const uint32_t a0 = tok_cnt;
      for (int t = 0; t < p.tiles; ++t) {
        const uint32_t idx = p.streaming ? a0 + (uint32_t)(p.tiles + t) : a0 + (uint32_t)t;
        const int s = (int)(idx & 1u);
        const int buf = (int)(d_cnt & 1u);
        wait_bar(d_full(buf), (d_cnt >> 1) & 1u);
        tc_fence_after();
        uint8_t* stp = sp + s * kStage;
        {
          float v[6][16];
          tmem_ld_cols<6>(tl + (uint32_t)(buf * 192 + hs * 96), v);
          tc_fence_before();
          mbar_arrive_warp(d_empty(buf));                    // accumulator is in registers: the next tile's MMAs may overwrite it
#pragma unroll
          if (row < p.TT) {                             // compact (resident) stages hold only TT rows per block
#pragma unroll
            for (int i = 0; i < 6; ++i) {
              const int c0 = hs * 96 + 16 * i;
              store16(stp + (c0 >> 6) * p.blk, row, (c0 & 63) >> 3, v[i]);
            }
          }
        }
        fence_proxy_async_smem();
        mbar_arrive_warp(st_ready(s));
        ++d_cnt;
      }
      tok_cnt = a0 + (uint32_t)(mult * p.tiles);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

// ---------------------------------------------------------------------------------------------------------
// weights-only operand images (run once per weight load)
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tile_token(const SccTile& g, int t, int r, int* ly, int* lx) {
  *ly = (t / g.tiles_x) * g.by + r / g.bx;
  *lx = (t % g.tiles_x) * g.bx + r % g.bx;
}
__device__ __forceinline__ size_t swz_elem(int row, int k) {      // byte offset of element k (< 64) of `row` in a SW128 block
  return (size_t)row * 128 + ((((k >> 3) ^ (row & 7))) << 4) + (k & 7) * 2;
}

__global__ void scc_pool_image_kernel(const float* __restrict__ wsl, int w, int base, uint8_t* __restrict__ img, int pool_bytes) {
  const SccTile g = scc_tile(w);
  const int r_ = w / base;
  const int kblocks = pool_bytes / 8192;
  const long long total = (long long)g.tiles * kblocks * 64 * 64;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(idx & 63); const int m = (int)((idx >> 6) & 63); const long long t2 = idx >> 12;
    const int kb = (int)(t2 % kblocks); const int t = (int)(t2 / kblocks);
    const int r = kb * 64 + k;
    float v = 0.f;
    if (r < g.TT && m < base * base) {
      int ly, lx; tile_token(g, t, r, &ly, &lx);
      if ((ly / r_) * base + lx / r_ == m) v = wsl[(ly % r_) * r_ + lx % r_];
    }
    *reinterpret_cast<bf16*>(img + (size_t)t * pool_bytes + (size_t)kb * 8192 + swz_elem(m, k)) = __float2bfloat16(v);
  }
}

// bias_tbl fp32 [6][L][Lb] (pack.cu pooled_bias_kernel, window-row-major tokens) -> per (tile, head) [TT rows][64 cells] SW128 images
__global__ void scc_bias_image_kernel(const float* __restrict__ tbl, int w, int base, uint8_t* __restrict__ img) {
  const SccTile g = scc_tile(w);
  const int L = w * w, Lb = base * base;
  const long long total = (long long)g.tiles * kHeads * g.TT * 64;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int m = (int)(idx & 63); long long t2 = idx >> 6;
    const int r = (int)(t2 % g.TT); t2 /= g.TT;
    const int h = (int)(t2 % kHeads); const int t = (int)(t2 / kHeads);
    int ly, lx; tile_token(g, t, r, &ly, &lx);
    const float v = m < Lb ? tbl[((long long)h * L + (ly * w + lx)) * Lb + m] : 0.f;
    *reinterpret_cast<bf16*>(img + ((size_t)t * kHeads + h) * (size_t)(g.TT * 128) + swz_elem(r, m)) = __float2bfloat16(v);
  }
}

// [16 rows o][64 k]: k<15: W1[o][k]/2, k==15: (bk1[o]+bk2[o])/2 (rides on the ones column of every head's q slice),
// 16<=k<31: W2[o][k-16]/2; row 15 = 0
__global__ void scc_w_image_kernel(const float* __restrict__ w1, const float* __restrict__ b1, const float* __restrict__ w2, const float* __restrict__ b2,
                                   uint8_t* __restrict__ img) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 16 * 64) return;
  const int o = idx >> 6, k = idx & 63;
  float v = 0.f;
  if (o < kHd) {
    if (k < kHd) v = 0.5f * w1[o * kHd + k];
    else if (k == 15) v = 0.5f * (b1[o] + b2[o]);
    else if (k >= 16 && k < 16 + kHd) v = 0.5f * w2[o * kHd + (k - 16)];
  }
  *reinterpret_cast<bf16*>(img + swz_elem(o, k)) = __float2bfloat16(v);
}

}  // namespace

size_t scc_pool_image_bytes(int w) { const SccTile g = scc_tile(w); return (size_t)g.tiles * (size_t)((g.TT > 64 ? g.TT / 64 : 1) * 8192); }
size_t scc_bias_image_bytes(int w) { const SccTile g = scc_tile(w); return (size_t)g.tiles * kHeads * (size_t)(g.TT * 128); }

int launch_scc_images(const SccW& w, int win, int base, uint8_t* pool_img, uint8_t* bias_img, uint8_t* w_img, cudaStream_t st) {
  const SccTile g = scc_tile(win);
  const int pool_bytes = (g.TT > 64 ? g.TT / 64 : 1) * 8192;
  if (pool_img != nullptr) {
    const long long total = (long long)g.tiles * (pool_bytes / 8192) * 4096;
    const int grid = (int)((total + 255) / 256 < 4096 ? (total + 255) / 256 : 4096);
    scc_pool_image_kernel<<<grid, 256, 0, st>>>(w.wsl, win, base, pool_img, pool_bytes);
    HITSIR_CHECK(cudaGetLastError());
  }
  {
    const long long total = (long long)g.tiles * kHeads * g.TT * 64;
    const int grid = (int)((total + 255) / 256 < 4096 ? (total + 255) / 256 : 4096);
    scc_bias_image_kernel<<<grid, 256, 0, st>>>(w.bias_tbl, win, base, bias_img);
    HITSIR_CHECK(cudaGetLastError());
  }
  scc_w_image_kernel<<<4, 256, 0, st>>>(w.wk1, w.bk1, w.wk2, w.bk2, w_img);
  HITSIR_CHECK(cudaGetLastError());
  return 0;
}

int launch_scc_umma(const bf16* t, const SccGeom& g, const SccW& w, bf16* out, int num_sms, cudaStream_t st) {
  static unsigned long long configured = 0;
  if (ensure_dynamic_smem(scc_umma_kernel, kSmemBytes, &configured)) return 1;
  const SccTile tg = scc_tile(g.w);
  if (tg.TT == 0) { set_error("launch_scc_umma: unsupported window %d", g.w); return 1; }
  Params p;
  p.nwin = g.pg.B * g.nWy * g.nWx; p.nWx = g.nWx; p.nWy = g.nWy;
  p.w = g.w; p.bx = tg.bx; p.by = tg.by; p.TT = tg.TT; p.tiles_x = tg.tiles_x; p.tiles = tg.tiles; p.ksteps = tg.TT / 16;
  p.Lb = g.Lb; p.streaming = tg.tiles > 2 ? 1 : 0;
  p.cell_ksteps = (g.Lb + 15) / 16;
  p.resident = tg.tiles == 1 ? 1 : 0;
  p.blk = p.resident ? tg.TT * 128 : kBlk;
  p.invL = 1.0f / (float)g.L;
  p.pool_bytes = (tg.TT > 64 ? tg.TT / 64 : 1) * 8192;
  p.bias_bytes = tg.TT * 128;
  p.pool_img = w.pool_img; p.bias_img = w.bias_img; p.w_img = w.w_img; p.bsl = w.bsl_dev;
  p.H = g.pg.H; p.W = g.pg.W;
  CUtensorMap tm_t, tm_o;
  if (make_tmap_nhwc(&tm_t, t, g.pg.B, g.pg.Hp, g.pg.Wp, kCp, 64, (uint32_t)tg.bx, (uint32_t)tg.by)) return 1;
  if (make_tmap_nhwc(&tm_o, out, g.pg.B, g.pg.H, g.pg.W, kCp, 64, (uint32_t)tg.bx, (uint32_t)tg.by)) return 1;
  const int grid = p.nwin < num_sms ? p.nwin : num_sms;
  HITSIR_CHECK(launch_pdl(scc_umma_kernel, dim3(grid), dim3(384), kSmemBytes, st, tm_t, tm_o, p));
  return 0;
}

}  // namespace hitsir
