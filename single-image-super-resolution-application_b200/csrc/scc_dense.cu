// Window self-correlation for the small windows (w = 4, 8; L = w*w <= 64 tokens, pooling ratio r = 1) on tcgen05:
// several windows share one 128-token tile and every per-window product becomes a block-diagonal ("masked") dense
// contraction over the tile, so the tensor core always works on M = 128 and nothing is ever reduced per window on its own.
// (SCC.forward without the final proj, /root/reference/models/hit_sir_pro.py:542-596; scc_umma.cu covers w >= 16.)
//
// With r = 1 the pooled keys/values are affine in the tokens: kp = a k + b, vp = a v + b (a = spatial_linear.weight, b = its
// bias, :451-455), and with no softmax the products re-associate per window (l, l', m = tokens of the window, L = w*w):
//   k-gen   K  = T Wk^T                                 12 MMAs (N=16)   -> bf16 K tile                     (:572)
//   C-SC    St = V K^T ;  P_c = mask(St) / L ;          6 + 8 MMAs       out_c = P_c Q  == (Q^T K / L) V^T   (:531,538)
//   S-SC    S_h = Q_h K_h^T ; P_h = mask((a S_h + b sum_i q_i) / 15 + bias_h) ;   out_s_h = a P_h V_h + b rowsum(P_h)
//                                                       6 x (1 + 8) MMAs                                    (:475,503,511)
// mask() keeps the L x L diagonal blocks; the off-diagonal parts of the P operands are zeroed once and never written.
// Token layout: head-padded 192 channels with ones in the q pads (kernels.cuh), so the k-gen bias rides in the contraction.
//
// Warp roles: 0 = TMA producer, 1 = MMA issuer, 2 = TMEM allocator, 3 = TMA store, 4..11 = converters.  The seven "score steps"
// of a tile (C-SC, heads 0..5) alternate between two TMEM score buffers / two P operand buffers, each owned by one converter
// group (hs = step & 1), so score MMA k+1, conversion k and output MMA k-1 overlap.
#include "gemm.cuh"
#include "kernels.cuh"

namespace hitsir {

namespace {

constexpr int kBlk = 16384;                 // [128 rows x 128 B] SWIZZLE_128B block
constexpr int kStage = 3 * kBlk;            // token tile: 3 channel blocks
constexpr int kOffK = 2 * kStage;           // bf16 K tile [128][96] (2 blocks)
constexpr int kOffP = kOffK + 2 * kBlk;     // 2 P operand buffers [128][128] (2 blocks each)
constexpr int kOffW = kOffP + 4 * kBlk;     // k-gen operand image (2 KB)
constexpr int kOffBias = kOffW + 2048;      // 2 slots x 8 KB: bf16 relative-position bias image of the head in flight (one per converter group)
constexpr int kOffBars = kOffBias + 2 * 8192;
constexpr int kNumBars = 24;
constexpr int kSmemBytes = kOffBars + kNumBars * 8 + 16 + 1024;
static_assert(kSmemBytes <= 232448, "smem budget");
constexpr int kTmS = 0;                     // score buffers at columns 0 and 128 (the k-gen accumulator aliases buffer 0)
constexpr int kTmD = 256;                   // output accumulator [128 x 192]

struct Params {
  int nwin, nWx, nWy, ntiles;
  int w, L, NW;              // window side, tokens per window, windows per 128-token tile
  const float* wsl;          // spatial_linear.weight[0] (r = 1)
  const float* bsl;          // spatial_linear.bias
  const uint8_t* bias_img;   // bf16 relative-position bias images [6][L rows][64 cells], 128-byte rows, SWIZZLE_128B chunk order
  int bias_bytes;            // L * 128
  const uint8_t* w_img;      // k-gen operand image (scc_umma.cu scc_w_image_kernel)
  int H, W;
};

// LT = tokens per window (16 or 64)
template <int LT>
__global__ void __launch_bounds__(384, 1)
scc_dense_kernel(const __grid_constant__ CUtensorMap tm_t, const __grid_constant__ CUtensorMap tm_o, const Params p) {
  constexpr int NW = 128 / LT;
  constexpr int NG = LT / 16;                  // 16-column groups of a window's diagonal block
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sb = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sp = smem_raw + (sb - smem_u32(smem_raw));
  const uint32_t bar0 = sb + kOffBars;
  auto tok_full = [&](int s) { return bar0 + 8u * s; };
  auto tok_empty = [&](int s) { return bar0 + 8u * (2 + s); };
  auto s_full = [&](int s) { return bar0 + 8u * (4 + s); };
  auto s_empty = [&](int s) { return bar0 + 8u * (6 + s); };
  auto p_full = [&](int s) { return bar0 + 8u * (8 + s); };
  auto p_empty = [&](int s) { return bar0 + 8u * (10 + s); };
  auto st_ready = [&](int s) { return bar0 + 8u * (12 + s); };
  auto b_full = [&](int s) { return bar0 + 8u * (18 + s); };
  auto b_empty = [&](int s) { return bar0 + 8u * (20 + s); };
  const uint32_t kt_full = bar0 + 8u * 14, k_ready = bar0 + 8u * 15, d_full = bar0 + 8u * 16, d_empty = bar0 + 8u * 17;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(sp + kOffBars + kNumBars * 8);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) { tma_prefetch_desc(&tm_t); tma_prefetch_desc(&tm_o); }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < 2; ++s) {
      mbar_init(tok_full(s), 1); mbar_init(tok_empty(s), 1);
      mbar_init(s_full(s), 1); mbar_init(s_empty(s), 4);
      mbar_init(p_full(s), 4); mbar_init(p_empty(s), 1);
      mbar_init(st_ready(s), 8);
      mbar_init(b_full(s), 1); mbar_init(b_empty(s), 4);
    }
    mbar_init(kt_full, 1); mbar_init(k_ready, 8); mbar_init(d_full, 1); mbar_init(d_empty, 8);
    fence_barrier_init();
  }
  if (warp == 2) { tmem_alloc(smem_u32(tmem_ptr_smem), 512); tmem_relinquish(); }
  // zero the token stages (rows of never-loaded windows must be finite) and the P operand buffers (off-diagonal blocks stay 0)
  for (int i = threadIdx.x; i < (kOffW) / 16; i += blockDim.x) reinterpret_cast<uint4*>(sp)[i] = make_uint4(0u, 0u, 0u, 0u);
  for (int i = threadIdx.x; i < 2048 / 16; i += blockDim.x)
    reinterpret_cast<uint4*>(sp + kOffW)[i] = reinterpret_cast<const uint4*>(p.w_img)[i];
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_ptr_smem;
  pdl_entry();                                           // up to here only the weights-only k-gen image was read

  if (warp == 0) {
    if (lane == 0) {
      // ===================== producer: one TMA box per (window, channel block); bias image of every head step =====================
      uint32_t cnt = 0, ub[2] = {0, 0};
      auto load_tile = [&](int tile, uint32_t c) {
        const int s = (int)(c & 1u);
        wait_bar(tok_empty(s), ((c >> 1) & 1u) ^ 1u);
        const int nvalid = min(NW, p.nwin - tile * NW);
        mbar_expect_tx(tok_full(s), (uint32_t)(nvalid * LT * 128 * 3));
        for (int i = 0; i < nvalid; ++i) {
          const int win = tile * NW + i;
          const int wx = win % p.nWx; const int t2 = win / p.nWx; const int wy = t2 % p.nWy; const int b = t2 / p.nWy;
#pragma unroll
          for (int blk = 0; blk < 3; ++blk)
            tma_load_4d(sb + s * kStage + blk * kBlk + i * LT * 128, &tm_t, tok_full(s), blk * 64, wx * p.w, wy * p.w, b);
        }
      };
      if (LT == 16) {          // all six 2 KB bias images fit the slot area: load them once
        mbar_expect_tx(b_full(0), (uint32_t)(kHeads * p.bias_bytes));
        bulk_load(sb + kOffBias, p.bias_img, (uint32_t)(kHeads * p.bias_bytes), b_full(0));
      }
      if ((int)blockIdx.x < p.ntiles) load_tile(blockIdx.x, 0);
      for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x, ++cnt) {
        if (tile + (int)gridDim.x < p.ntiles) load_tile(tile + gridDim.x, cnt + 1);     // tokens run one tile ahead
        if (LT == 16) continue;
        for (int k = 1; k <= kHeads; ++k) {
          const int slot = k & 1;
          wait_bar(b_empty(slot), (ub[slot] & 1u) ^ 1u);
          mbar_expect_tx(b_full(slot), (uint32_t)p.bias_bytes);
          bulk_load(sb + kOffBias + slot * 8192, p.bias_img + (size_t)(k - 1) * p.bias_bytes, (uint32_t)p.bias_bytes, b_full(slot));
          ++ub[slot];
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ===================== MMA issuer =====================
      constexpr uint32_t id_k16 = make_idesc(128, 16, 0, 0);     // k-gen: T_h Wk^T
      constexpr uint32_t id_s = make_idesc(128, 128, 0, 0);      // scores: (V | Q_h) K^T
      constexpr uint32_t id_oc = make_idesc(128, 96, 0, 1);      // out_c = P_c Q   (B = token tile, MN-major)
      constexpr uint32_t id_os = make_idesc(128, 16, 0, 1);      // out_s_h = P_h V_h
      const uint32_t kb = sb + kOffK, wb = sb + kOffW;
      const uint64_t w1d = umma_desc_sw128(wb), w2d = umma_desc_sw128(wb + 32);
      uint32_t cnt = 0, us[2] = {0, 0}, up[2] = {0, 0};
      for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x, ++cnt) {
        const int s = (int)(cnt & 1u);
        const uint32_t st = sb + s * kStage;
        wait_bar(tok_full(s), (cnt >> 1) & 1u);
        wait_bar(s_empty(0), (us[0] & 1u) ^ 1u);         // the k-gen accumulator aliases score buffer 0
        tc_fence_after();
        // ---- k-gen: K[:, 16h..] = Q_h W1^T (+ bias via the ones column) + V_h W2^T
#pragma unroll
        for (int h = 0; h < kHeads; ++h) umma_bf16(tmem + kTmS + 16 * h, umma_desc_sw128(st + (h >> 2) * kBlk + (h & 3) * 32), w1d, id_k16, 0u);
#pragma unroll
        for (int h = 0; h < kHeads; ++h) {
          const int cv = 96 + 16 * h;
          umma_bf16(tmem + kTmS + 16 * h, umma_desc_sw128(st + (cv >> 6) * kBlk + (cv & 63) * 2), w2d, id_k16, 1u);
        }
        umma_commit(kt_full);
        wait_bar(k_ready, cnt & 1u);
        tc_fence_after();
        auto out_step = [&](int j) {
          const int buf = j & 1;
          wait_bar(p_full(buf), up[buf] & 1u);
          if (j == 0) wait_bar(d_empty, (cnt & 1u) ^ 1u);
          tc_fence_after();
          const uint32_t pb = sb + kOffP + buf * 2 * kBlk;
          if (j == 0) {
#pragma unroll
            for (int ks = 0; ks < 8; ++ks)
              umma_bf16(tmem + kTmD + 96, umma_desc_sw128(pb + (ks >> 2) * kBlk + (ks & 3) * 32), make_desc(st + ks * 2048, kBlk, 1024), id_oc, ks ? 1u : 0u);
          } else {
            const int h = j - 1, cv = 96 + 16 * h;
            const uint32_t vb = st + (cv >> 6) * kBlk + (cv & 63) * 2;
#pragma unroll
            for (int ks = 0; ks < 8; ++ks)
              umma_bf16(tmem + kTmD + 16 * h, umma_desc_sw128(pb + (ks >> 2) * kBlk + (ks & 3) * 32), make_desc(vb + ks * 2048, kBlk, 1024), id_os, ks ? 1u : 0u);
          }
          umma_commit(p_empty(buf));
          ++up[buf];
        };
        for (int k = 0; k <= kHeads; ++k) {
          const int buf = k & 1;
          wait_bar(s_empty(buf), (us[buf] & 1u) ^ 1u);
          tc_fence_after();
          const uint32_t S = tmem + kTmS + 128 * buf;
          if (k == 0) {
#pragma unroll
            for (int ks = 0; ks < 6; ++ks) {             // St[l][l'] = sum_c v_l[c] k_l'[c]
              const int cv = 96 + 16 * ks;
              umma_bf16(S, umma_desc_sw128(st + (cv >> 6) * kBlk + (cv & 63) * 2), umma_desc_sw128(kb + (ks >> 2) * kBlk + (ks & 3) * 32), id_s, ks ? 1u : 0u);
            }
          } else {
            const int h = k - 1;                         // S_h[l][m] = q_lh . k_mh
            umma_bf16(S, umma_desc_sw128(st + (h >> 2) * kBlk + (h & 3) * 32), umma_desc_sw128(kb + (h >> 2) * kBlk + (h & 3) * 32), id_s, 0u);
          }
          umma_commit(s_full(buf));
          ++us[buf];
          if (k >= 1) out_step(k - 1);
        }
        out_step(kHeads);
        umma_commit(d_full);
      }
    }
  } else if (warp == 3) {
    if (lane == 0) {
      // ===================== TMA store, one box per (window, channel block) =====================
      uint32_t cnt = 0;
      for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x, ++cnt) {
        const int s = (int)(cnt & 1u);
        wait_bar(st_ready(s), (cnt >> 1) & 1u);
        const int nvalid = min(NW, p.nwin - tile * NW);
        bool any = false;
        for (int i = 0; i < nvalid; ++i) {
          const int win = tile * NW + i;
          const int wx = win % p.nWx; const int t2 = win / p.nWx; const int wy = t2 % p.nWy; const int b = t2 / p.nWy;
          if (wx * p.w < p.W && wy * p.w < p.H) {       // windows entirely inside the reflect padding are cropped (:696)
#pragma unroll
            for (int blk = 0; blk < 3; ++blk)
              tma_store_4d(&tm_o, sb + s * kStage + blk * kBlk + i * LT * 128, blk * 64, wx * p.w, wy * p.w, b);
            any = true;
          }
        }
        if (any) { tma_commit(); tma_wait_read<0>(); }
        mbar_arrive(tok_empty(s));
      }
      tma_wait_all0();
    }
  } else if (warp >= 4) {
    // ===================== converters (8 warps): thread = (token row, group hs) =====================
    const int q = warp & 3, hs = (warp - 4) >> 2;
    const int row = q * 32 + lane;
    const int wl = row / LT, l_loc = row % LT;
    const uint32_t tl = tmem + ((uint32_t)(q * 32) << 16);
    const float a = p.wsl[0], b = *p.bsl;
    // TMEM columns of this warp's diagonal block(s): L=16 -> both windows of the warp (32 columns, lane picks its half)
    const int colbase = (LT == 16) ? 32 * q : LT * wl;
    uint8_t* pbuf = sp + kOffP + hs * 2 * kBlk;
    uint32_t cnt = 0, u = 0, ubias = 0;
    uint8_t* bslot = sp + kOffBias + hs * 8192;
    if (LT == 16) wait_bar(b_full(0), 0u);
    for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x, ++cnt) {
      const int s = (int)(cnt & 1u);
      uint8_t* stp = sp + s * kStage;
      // ---- K tile: accumulator columns [48 hs, 48 hs + 48) -> bf16
      wait_bar(kt_full, cnt & 1u);
      tc_fence_after();
      {
        float v[3][16];
        tmem_ld_cols<3>(tl + kTmS + hs * 48, v);
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          const int c0 = hs * 48 + 16 * i;
          store16(sp + kOffK + (c0 >> 6) * kBlk, row, (c0 & 63) >> 3, v[i]);
        }
      }
      tc_fence_before();
      fence_proxy_async_smem();
      mbar_arrive_warp(k_ready);
      float rowsum[3] = {0.f, 0.f, 0.f};
      // ---- score steps of this group: k = hs, hs + 2, ...  (k = 0: C-SC, k >= 1: head k - 1)
#pragma unroll 1
      for (int k = hs; k <= kHeads; k += 2, ++u) {
        wait_bar(s_full(hs), u & 1u);
        tc_fence_after();
        float sc[(LT == 16) ? 2 : NG][16];
        tmem_ld_cols<(LT == 16) ? 2 : NG>(tl + kTmS + 128 * hs + colbase, sc);
        tc_fence_before();
        mbar_arrive_warp(s_empty(hs));
        // this row's diagonal block (L = 16: pick the warp half that holds this row's window)
        float base[NG][16];
#pragma unroll
        for (int g = 0; g < NG; ++g)
#pragma unroll
          for (int e = 0; e < 16; ++e) base[g][e] = (LT == 16) ? ((lane & 16) ? sc[1][e] : sc[0][e]) : sc[(LT == 16) ? 0 : g][e];
        float val[NG][16];
        if (k == 0) {
#pragma unroll
          for (int g = 0; g < NG; ++g)
#pragma unroll
            for (int e = 0; e < 16; ++e) val[g][e] = base[g][e] * (1.0f / (float)LT);
        } else {
          const int h = k - 1;
          // sum_i q_l[(h,i)], i < 15, from this token's row of the tile
          const int pc = (16 * h) & 63;
          uint8_t* blkp = stp + ((16 * h) >> 6) * kBlk;
          const uint4 q0 = *reinterpret_cast<const uint4*>(swz(blkp, row, pc >> 3));
          const uint4 q1 = *reinterpret_cast<const uint4*>(swz(blkp, row, (pc >> 3) + 1));
          const uint32_t qw[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
          float qsum = 0.f;
#pragma unroll
          for (int i = 0; i < 8; ++i) { const float2 f = unpack_bf16x2(qw[i]); qsum += f.x + (i == 7 ? 0.f : f.y); }
          const float add = b * qsum * (1.0f / 15.0f), mul = a * (1.0f / 15.0f);
          if (LT == 16) bslot = sp + kOffBias + h * 2048;
          else wait_bar(b_full(hs), ubias & 1u);
          float rs = 0.f;
#pragma unroll
          for (int g = 0; g < NG; ++g) {
            const uint4 b0 = *reinterpret_cast<const uint4*>(swz(bslot, l_loc, 2 * g));
            const uint4 b1 = *reinterpret_cast<const uint4*>(swz(bslot, l_loc, 2 * g + 1));
            const uint32_t bw[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int e = 0; e < 16; e += 2) {
              const float2 bb = unpack_bf16x2(bw[e >> 1]);
              val[g][e] = fmaf(mul, base[g][e], add) + bb.x;
              val[g][e + 1] = fmaf(mul, base[g][e + 1], add) + bb.y;
              rs += val[g][e] + val[g][e + 1];
            }
          }
          if (LT != 16) { mbar_arrive_warp(b_empty(hs)); ++ubias; }
          rowsum[(k - 1) >> 1] = rs;
        }
        wait_bar(p_empty(hs), (u & 1u) ^ 1u);
#pragma unroll
        for (int g = 0; g < NG; ++g) {
          const int col = wl * LT + 16 * g;              // diagonal block of this row's window
          store16(pbuf + (col >> 6) * kBlk, row, (col & 63) >> 3, val[g]);
        }
        fence_proxy_async_smem();
        mbar_arrive_warp(p_full(hs));
      }
      // ---- epilogue: out_s columns of this group's heads (a D + b rowsum) and half of out_c, in place over the token tile
      wait_bar(d_full, cnt & 1u);
      tc_fence_after();
      {
        float vs[3][16], vc[3][16];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          uint32_t r[16];
          tmem_ld16_nw(tl + kTmD + 16 * (2 * i + 1 - hs), r);      // hs = 0 owns heads 1,3,5 (steps 2,4,6); hs = 1 heads 0,2,4
          tmem_ld_wait();
          reg_fence16(r);
#pragma unroll
          for (int e = 0; e < 16; ++e) vs[i][e] = __uint_as_float(r[e]);
        }
        tmem_ld_cols<3>(tl + kTmD + 96 + 48 * hs, vc);
        tc_fence_before();
        mbar_arrive_warp(d_empty);
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          const int h = 2 * i + 1 - hs;
          // rowsum slot of head h inside this group: steps k = h + 1 -> index (k - 1) >> 1 = h >> 1
          const float add = b * rowsum[h >> 1];
#pragma unroll
          for (int e = 0; e < 16; ++e) vs[i][e] = fmaf(a, vs[i][e], add);
          store16(stp + ((16 * h) >> 6) * kBlk, row, ((16 * h) & 63) >> 3, vs[i]);
          const int c0 = 96 + 48 * hs + 16 * i;
          store16(stp + (c0 >> 6) * kBlk, row, (c0 & 63) >> 3, vc[i]);
        }
      }
      fence_proxy_async_smem();
      mbar_arrive_warp(st_ready(s));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

template <int LT>
int launch_lt(const CUtensorMap& tm_t, const CUtensorMap& tm_o, const Params& p, int num_sms, cudaStream_t st) {
  static unsigned long long configured = 0;
  if (ensure_dynamic_smem(scc_dense_kernel<LT>, kSmemBytes, &configured)) return 1;
  const int grid = p.ntiles < num_sms ? p.ntiles : num_sms;
  HITSIR_CHECK(launch_pdl(scc_dense_kernel<LT>, dim3(grid), dim3(384), kSmemBytes, st, tm_t, tm_o, p));
  return 0;
}

}  // namespace

int launch_scc_dense(const bf16* t, const SccGeom& g, const SccW& w, bf16* out, int num_sms, cudaStream_t st) {
  if (g.r != 1 || (g.L != 16 && g.L != 64)) { set_error("launch_scc_dense: window %d not supported", g.w); return 1; }
  Params p;
  p.nwin = g.pg.B * g.nWy * g.nWx; p.nWx = g.nWx; p.nWy = g.nWy;
  p.w = g.w; p.L = g.L; p.NW = 128 / g.L;
  p.ntiles = (p.nwin + p.NW - 1) / p.NW;
  p.wsl = w.wsl; p.bsl = w.bsl_dev; p.bias_img = w.bias_img; p.bias_bytes = g.L * 128; p.w_img = w.w_img;
  p.H = g.pg.H; p.W = g.pg.W;
  CUtensorMap tm_t, tm_o;
  if (make_tmap_nhwc(&tm_t, t, g.pg.B, g.pg.Hp, g.pg.Wp, kCp, 64, (uint32_t)g.w, (uint32_t)g.w)) return 1;
  if (make_tmap_nhwc(&tm_o, out, g.pg.B, g.pg.H, g.pg.W, kCp, 64, (uint32_t)g.w, (uint32_t)g.w)) return 1;
  return g.L == 16 ? launch_lt<16>(tm_t, tm_o, p, num_sms, st) : launch_lt<64>(tm_t, tm_o, p, num_sms, st);
}

}  // namespace hitsir
