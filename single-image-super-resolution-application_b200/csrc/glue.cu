// Bandwidth-bound glue kernels of the HiT-SIR-pro forward (everything that is not a dense
// contraction or the window self-correlation): entry im2col, LayerNorm, casa
// (SpatialChannelAttention) statistics and gating, UnionAttention/Fusion statistics and
// gating, nearest upsampling.  Token-major (NHWC) throughout; 128-bit accesses where rows allow.
#include "gemm.cuh"
#include "kernels.cuh"

namespace hitsir {

namespace {

// ---------------------------------------------------------------------------------------------
// Entry: mean shift (:1310-1311) + im2col of the f x f footprint.  CTA = (image, row, run of 64 pixels): the f rows x (64 + f - 1)
// columns x in_ch window is staged once in shared memory as bf16((x - mean) * img_range) (zero outside the image = the conv's zero
// padding), a table maps every K index to its offset in that window, and a warp then writes whole 2*Kp-byte im2col rows (one 16-byte
// chunk per lane).  The first version recomputed tap / channel / bounds per output element with scattered global loads: 2.4 ms at
// cfg2 for 1 GB of output; this one is bound by the write.
constexpr int kImSeg = 64;
constexpr int kImMaxWin = 3 * 9 * (kImSeg + 8);
__global__ void __launch_bounds__(256) entry_im2col_kernel(const float* __restrict__ x, bf16* __restrict__ a0, int B, int H, int W, int in_ch, int f, int Kp,
                                                            float m0, float m1, float m2, float img_range, int nseg, int yb0, int Hf) {
  __shared__ bf16 tile[kImMaxWin];
  __shared__ uint16_t ktab[512];
  const int seg = blockIdx.x % nseg; const int t2 = blockIdx.x / nseg;
  const int y = t2 % H, b = t2 / H;
  const int x0 = seg * kImSeg, npx = min(kImSeg, W - x0);
  const int half = f / 2, kreal = f * f * in_ch, wcols = kImSeg + f - 1;
  for (int k = threadIdx.x; k < Kp; k += blockDim.x) {
    uint16_t off = 0xFFFFu;
    if (k < kreal) { const int tap = k / in_ch, c = k - tap * in_ch; off = (uint16_t)((c * f + tap / f) * wcols + tap % f); }
    ktab[k] = off;
  }
  for (int i = threadIdx.x; i < in_ch * f * wcols; i += blockDim.x) {
    const int cx = i % wcols; const int r2 = i / wcols; const int ry = r2 % f, c = r2 / f;
    const int yy = yb0 + y + ry - half, xx = x0 + cx - half;              // frame row (band mode: yb0 = first frame row of the band)
    float val = 0.f;
    if (yy >= 0 && yy < Hf && xx >= 0 && xx < W) {
      const float mean = (in_ch == 3) ? (c == 0 ? m0 : (c == 1 ? m1 : m2)) : 0.f;
      val = (__ldg(x + (((long long)b * in_ch + c) * Hf + yy) * W + xx) - mean) * img_range;
    }
    tile[i] = __float2bfloat16(val);
  }
  __syncthreads();
  const int chunks = Kp / 8;
  const uint16_t* tl = reinterpret_cast<const uint16_t*>(tile);
  bf16* row0 = a0 + (((long long)b * H + y) * W + x0) * Kp;
  for (int idx = threadIdx.x; idx < npx * chunks; idx += blockDim.x) {
    const int ch = idx % chunks, px = idx / chunks;
    uint32_t w[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const uint16_t o0 = ktab[ch * 8 + 2 * e], o1 = ktab[ch * 8 + 2 * e + 1];
      const uint32_t lo = o0 == 0xFFFFu ? 0u : (uint32_t)tl[o0 + px], hi = o1 == 0xFFFFu ? 0u : (uint32_t)tl[o1 + px];
      w[e] = lo | (hi << 16);
    }
    *reinterpret_cast<uint4*>(row0 + (long long)px * Kp + ch * 8) = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

// one warp per row
__global__ void ln_rows_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                               bf16* __restrict__ ob, float* __restrict__ of, long long N, const float* __restrict__ add, long long add_rows) {
  const int lane = threadIdx.x & 31;
  const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long row = warp0; row < N; row += nwarps) {
    const float* r = x + row * kC;
    float v[6];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 6; ++i) { const int c = lane + 32 * i; v[i] = c < kC ? r[c] : 0.f; s += v[i]; }
    const float mean = warp_sum(s) / (float)kC;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < 6; ++i) { const int c = lane + 32 * i; const float d = c < kC ? v[i] - mean : 0.f; q += d * d; }
    const float rstd = rsqrtf(warp_sum(q) / (float)kC + 1e-5f);
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      const int c = lane + 32 * i;
      float y = c < kC ? (v[i] - mean) * rstd * gamma[c] + beta[c] : 0.f;
      if (add != nullptr && c < kC) y += add[(row % add_rows) * kC + c];       // absolute position embedding, broadcast over the batch (:1293-1294)
      if (ob != nullptr) ob[row * kCp + c] = __float2bfloat16(y);
      if (of != nullptr && c < kC) of[row * kC + c] = y;
    }
  }
}

// PIL-style uint8 HWC image -> [0,1] fp32 NCHW (torchvision to_tensor: true division by 255; reference utils/utils.py:143-145)
__global__ void u8hwc_to_f32nchw_kernel(const uint8_t* __restrict__ in, float* __restrict__ out, int B, int H, int W, int C) {
  const long long total = (long long)B * C * H * W;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int x = (int)(i % W); long long t = i / W; const int y = (int)(t % H); t /= H; const int c = (int)(t % C); const int b = (int)(t / C);
    out[i] = (float)in[(((long long)b * H + y) * W + x) * C + c] / 255.0f;
  }
}
// fp32 NCHW -> clip(0,1) (experiments/experiment.py:746-748, test_experiment.py:75) -> uint8 HWC with to_pil_image's mul(255).byte() truncation,
// or (Round) with BasicSR's tensor2img (basicsr/utils/img_util.py): (v * 255.0).round() in fp32, half to even
template <bool Round>
__global__ void f32nchw_to_u8hwc_kernel(const float* __restrict__ in, uint8_t* __restrict__ out, int B, int H, int W, int C) {
  const long long total = (long long)B * H * W * C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C); long long t = i / C; const int x = (int)(t % W); t /= W; const int y = (int)(t % H); const int b = (int)(t / H);
    const float v = fminf(fmaxf(in[(((long long)b * C + c) * H + y) * W + x], 0.f), 1.f);
    out[i] = Round ? (uint8_t)rintf(__fmul_rn(v, 255.0f)) : (uint8_t)(v * 255.0f);
  }
}

__global__ void tap_kernel(const void* src, int is_bf16, int ld, float* dst, long long rows, int cols, int perm) {
  const long long total = rows * cols;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / cols; const int c0 = (int)(i - r * cols);
    const int c = perm ? scc_pos(c0) : c0;
    dst[i] = is_bf16 ? __bfloat162float(reinterpret_cast<const bf16*>(src)[r * ld + c]) : reinterpret_cast<const float*>(src)[r * ld + c];
  }
}

// bf16 [N,192] shadow (pad 0) of an fp32 [N,180] stream: thread = (row, 8 channels)
__global__ void cast_rows_bf16_kernel(const float* __restrict__ a, bf16* __restrict__ out, long long N) {
  constexpr int groups = kCp / 8;
  const long long total = N * groups;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / groups; const int c0 = (int)(i - r * groups) * 8;
    float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (c0 < kC) {
      const float4 v0 = *reinterpret_cast<const float4*>(a + r * kC + c0);
      v[0] = v0.x; v[1] = v0.y; v[2] = v0.z; v[3] = v0.w;
      if (c0 + 4 < kC) { const float4 v1 = *reinterpret_cast<const float4*>(a + r * kC + c0 + 4); v[4] = v1.x; v[5] = v1.y; v[6] = v1.z; v[7] = v1.w; }
    }
    *reinterpret_cast<uint4*>(out + r * kCp + c0) =
        make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
  }
}

__global__ void add_to_bf16_kernel(const float* __restrict__ a, const float* __restrict__ b, bf16* __restrict__ out, long long N) {
  const long long total = N * kCp;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / kCp; const int c = (int)(i - r * kCp);
    out[i] = __float2bfloat16(c < kC ? a[r * kC + c] + b[r * kC + c] : 0.f);
  }
}

// ---------------------------------------------------------------------------------------------
// casa statistics.  grid = (nparts, B); each CTA walks a slice of the padded map of one image,
// one warp per padded pixel, and emits a deterministic partial (sum, max) per channel.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) sca_stats_kernel(const float* __restrict__ x, PadGeom g, float* __restrict__ cavg, float* __restrict__ cmax,
                                                        float* __restrict__ part_sum, float* __restrict__ part_max, int nparts) {
  // cavg / cmax are stored for the UNPADDED pixels (the casa gate gathers them through the reflect map); the global pools run over
  // the reflect-padded map (:348-349 on the padded x of :554-557), i.e. every pixel counts once per padded position that mirrors it.
  __shared__ float s_sum[8][kCp];
  __shared__ float s_max[8][kCp];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.y, part = blockIdx.x;
  const int npix = g.H * g.W;
  const int per = (npix + nparts - 1) / nparts;
  const int p0 = part * per, p1 = min(npix, p0 + per);
  float asum[6], amax[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) { asum[i] = 0.f; amax[i] = -INFINITY; }
  // four pixels per warp iteration: 24 independent loads in flight before the shuffle reductions
  for (int pp0 = p0 + warp * 4; pp0 < p1; pp0 += 32) {
    float v[4][6];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int pp = min(pp0 + u, p1 - 1);
      const float* r = x + ((long long)b * npix + pp) * kC;
#pragma unroll
      for (int i = 0; i < 6; ++i) { const int c = lane + 32 * i; v[u][i] = c < kC ? r[c] : 0.f; }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int pp = pp0 + u;
      if (pp >= p1) break;
      const int y = pp / g.W, xw = pp - y * g.W;
      const float mult = (float)(reflect_mult(y + g.y0, g.Hf > 0 ? g.Hf : g.H, g.Hf > 0 ? g.Hpf : g.Hp) * reflect_mult(xw, g.W, g.Wp));
      float s = 0.f, m = -INFINITY;
#pragma unroll
      for (int i = 0; i < 6; ++i) {
        const int c = lane + 32 * i;
        if (c < kC) { s += v[u][i]; m = fmaxf(m, v[u][i]); asum[i] = fmaf(mult, v[u][i], asum[i]); amax[i] = fmaxf(amax[i], v[u][i]); }
      }
      s = warp_sum(s); m = warp_max(m);
      if (lane == 0) { cavg[(long long)b * npix + pp] = s / (float)kC; cmax[(long long)b * npix + pp] = m; }
    }
  }
#pragma unroll
  for (int i = 0; i < 6; ++i) { s_sum[warp][lane + 32 * i] = asum[i]; s_max[warp][lane + 32 * i] = amax[i]; }
  __syncthreads();
  if (threadIdx.x < kC) {
    float s = 0.f, m = -INFINITY;
#pragma unroll
    for (int wv = 0; wv < 8; ++wv) { s += s_sum[wv][threadIdx.x]; m = fmaxf(m, s_max[wv][threadIdx.x]); }
    part_sum[((long long)b * nparts + part) * kC + threadIdx.x] = s;
    part_max[((long long)b * nparts + part) * kC + threadIdx.x] = m;
  }
}

// one CTA per image: finish the global pools, then Linear C->18->C twice (no activation, :350-355).  768 threads: the partials are summed
// by four groups of 192 channel threads (fixed order within a group, groups merged in order), the 36 length-180 dot products of the first
// linears take one warp each (fixed shuffle tree): deterministic, and the serial chains that made this launch 54 us long are gone.
__global__ void __launch_bounds__(768) sca_mlp_kernel(const float* __restrict__ part_sum, const float* __restrict__ part_max, int nparts, PadGeom g,
                                                      CasaW w, float* __restrict__ s1, float* __restrict__ s2) {
  __shared__ float ps[4][kCp], pm[4][kCp], avg[kC], mx[kC], h1[18], h2[18];
  pdl_entry();
  const int b = blockIdx.x, grp = threadIdx.x / 192, c = threadIdx.x - grp * 192;
  if (c < kC) {
    float s = 0.f, m = -INFINITY;
    for (int p = grp; p < nparts; p += 4) { s += part_sum[((long long)b * nparts + p) * kC + c]; m = fmaxf(m, part_max[((long long)b * nparts + p) * kC + c]); }
    ps[grp][c] = s; pm[grp][c] = m;
  }
  __syncthreads();
  if (grp == 0 && c < kC) {
    avg[c] = (((ps[0][c] + ps[1][c]) + ps[2][c]) + ps[3][c]) / (float)((g.Hf > 0 ? g.Hpf : g.Hp) * g.Wp);
    mx[c] = fmaxf(fmaxf(pm[0][c], pm[1][c]), fmaxf(pm[2][c], pm[3][c]));
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int o = warp; o < 36; o += 24) {                    // outputs 0..17: linear1_first on the average pool, 18..35: linear2_first on the max pool
    const int j = o % 18;
    const float* wr = (o < 18 ? w.l1f_w : w.l2f_w) + j * kC;
    const float* v = o < 18 ? avg : mx;
    float a = 0.f;
    for (int k = lane; k < kC; k += 32) a = fmaf(wr[k], v[k], a);
    a = warp_sum(a);
    if (lane == 0) { if (o < 18) h1[j] = a + w.l1f_b[j]; else h2[j] = a + w.l2f_b[j]; }
  }
  __syncthreads();
  if (grp == 0 && c < kC) {
    float a = w.l1s_b[c], bb = w.l2s_b[c];
#pragma unroll
    for (int k = 0; k < 18; ++k) { a += w.l1s_w[c * 18 + k] * h1[k]; bb += w.l2s_w[c * 18 + k] * h2[k]; }
    s1[(long long)b * kC + c] = a; s2[(long long)b * kC + c] = bb;
  }
}

// thread = (padded pixel, 8 head-padded positions); no casa gate (Identity qkv, :552)
__global__ void qkv_build_kernel(const float* __restrict__ x, PadGeom g, bf16* __restrict__ t) {
  constexpr int groups = kCp / 8;   // 24
  const long long total = (long long)g.B * g.Hp * g.Wp * groups;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int gi = (int)(idx % groups);
    const long long pix = idx / groups;
    const int xp = (int)(pix % g.Wp); const long long tt = pix / g.Wp; const int yp = (int)(tt % g.Hp); const int b = (int)(tt / g.Hp);
    const float* r = x + (((long long)b * g.H + reflect_src(yp, g.H)) * g.W + reflect_src(xp, g.W)) * kC;
    float o[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int pos = gi * 8 + e, c = scc_chan(pos);
      o[e] = c >= 0 ? r[c] : (pos < 96 ? 1.0f : 0.f);       // q pads carry the constant 1 (k-gen bias rider), v pads 0
    }
    *reinterpret_cast<uint4*>(t + pix * kCp + gi * 8) =
        make_uint4(pack_bf16x2(o[0], o[1]), pack_bf16x2(o[2], o[3]), pack_bf16x2(o[4], o[5]), pack_bf16x2(o[6], o[7]));
  }
}

// ---------------------------------------------------------------------------------------------
// casa gate on the tensor core.  The two Conv2d(1, C, 3) of SpatialChannelAttention (:345-347) are a K = 9 contraction per pixel
// and channel: 18 FP32 FMAs per output, which made a SIMT version of this kernel FMA/issue-bound at 2.8 TB/s.  Here they are
// warp-level bf16 MMAs (m16n8k16, fp32 accumulate) with a three-term split so that nothing is lost to bf16:
//     k  0.. 8: a_hi[tap] * W_hi[tap]      k  9..17: a_lo[tap] * W_hi[tap]      k 18..26: a_hi[tap] * W_lo[tap]
//     k 27, 28: 1 * b_hi, 1 * b_lo         k 29..31: 0                          (x = x_hi + x_lo, both bf16: ~16 mantissa bits)
// CTA = (image, padded row), 4 warps, 5 CTAs per SM (96 registers); per run of 32 padded pixels: the token rows are staged by ONE bulk copy (the
// pixels of a run are contiguous in global memory; only the reflected tail of a padded row goes pixel by pixel) that completes on an
// mbarrier -- per-thread 16-byte cp.async chunks (45 per row) ran at 4.0 TB/s, the bulk copy at 4.7 --, every warp owns 6 n-tiles
// (48 head-padded positions) whose B fragments stay in registers for the whole row, the A
// rows [32 px][32 k] of both statistic maps are built once per run in shared memory, and the gated bf16 tokens leave through a
// padded shared tile as one 384-byte bulk store per pixel (per-thread 16-byte stores: 18.8 -> 17.9 ms/step).  What is left per output: 2 LeakyReLU, 2 FMA, the token read and the bf16 pack.
constexpr int kQkvMinCtas = 5;                   // 96 registers, no spills: shared memory (43 KB per CTA) then allows 5 CTAs per SM instead of 3 at 140 registers
constexpr int kMmaRun = 32;
constexpr int kMmaXS = 180;                      // staged token rows keep their global pitch (720 B): a run of pixels is ONE bulk copy
constexpr int kMmaOS = 100;                      // output row: 96 words + 4 (rows of a quad-store land on distinct banks)
constexpr int kMmaAS = 20;                       // A row: 16 words + 4
constexpr int kMmaSmem = kMmaRun * kMmaXS * 4 + kMmaRun * kMmaOS * 4 + 2 * kMmaRun * kMmaAS * 4 + 2 * kCp * 4 + 2 * 3 * (kMmaRun + 2) * 4;
constexpr int kCasaBfragWords = 24 * 2 * 2 * 2 * 32;

__device__ __forceinline__ void split_bf16(float v, uint16_t* hi, uint16_t* lo) {
  const bf16 h = __float2bfloat16_rn(v);
  const bf16 l = __float2bfloat16_rn(v - __bfloat162float(h));
  *hi = *reinterpret_cast<const uint16_t*>(&h); *lo = *reinterpret_cast<const uint16_t*>(&l);
}
// B fragments of both 3x3 filters in the k order above: img[n-tile 24][conv 2][k-step 2][reg 2][lane 32]
__global__ void casa_bfrag_kernel(CasaW w, uint32_t* __restrict__ img) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= kCasaBfragWords) return;
  const int lane = idx & 31, i = (idx >> 5) & 1, s = (idx >> 6) & 1, v = (idx >> 7) & 1, nt = idx >> 8;
  const int c = scc_chan(nt * 8 + (lane >> 2));
  const float* wt = v == 0 ? w.w1 : w.w2;
  const float* bs = v == 0 ? w.b1 : w.b2;
  uint16_t out[2];
#pragma unroll
  for (int e = 0; e < 2; ++e) {
    const int k = s * 16 + i * 8 + (lane & 3) * 2 + e;
    uint16_t hi = 0, lo = 0, r = 0;
    if (c >= 0) {
      if (k < 27) { split_bf16(wt[(k % 9) * kC + c], &hi, &lo); r = k < 18 ? hi : lo; }
      else if (k < 29) { split_bf16(bs[c], &hi, &lo); r = k == 27 ? hi : lo; }
    }
    out[e] = r;
  }
  img[idx] = (uint32_t)out[0] | ((uint32_t)out[1] << 16);
}

__global__ void __launch_bounds__(128, kQkvMinCtas) qkv_casa_mma_kernel(const float* __restrict__ x, PadGeom g, const float* __restrict__ cavg,
                                                           const float* __restrict__ cmax, const float* __restrict__ s1, const float* __restrict__ s2,
                                                           const uint32_t* __restrict__ bfrag, bf16* __restrict__ t) {
  pdl_entry();
  extern __shared__ __align__(16) uint8_t smem_casa[];
  float* xs = reinterpret_cast<float*>(smem_casa);                       // [run][184]
  uint32_t* os = reinterpret_cast<uint32_t*>(xs + kMmaRun * kMmaXS);     // [run][100]
  uint32_t* as = os + kMmaRun * kMmaOS;                                  // [2][run][20]
  float* gs = reinterpret_cast<float*>(as + 2 * kMmaRun * kMmaAS);       // [2][192]: 0.5 * channel gate in head-padded order (0 on pads)
  float* sw = gs + 2 * kCp;                                              // [2][3][run + 2] statistic windows
  const int yp = blockIdx.x % g.Hp, b = blockIdx.x / g.Hp;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, gq = lane >> 2, tq = lane & 3;
  const int ysrc = reflect_src(yp, g.H);
  const float* xrow = x + ((long long)b * g.H + ysrc) * g.W * kC;
  const float* ca = cavg + (long long)b * g.H * g.W;
  const float* cm = cmax + (long long)b * g.H * g.W;
  const uint32_t xs_addr = (uint32_t)__cvta_generic_to_shared(xs);
  __shared__ __align__(8) uint64_t xbar_storage;
  const uint32_t xbar = (uint32_t)__cvta_generic_to_shared(&xbar_storage);
  if (tid == 0) { mbar_init(xbar, 1); fence_barrier_init(); }
  __syncthreads();
  uint32_t xphase = 0;
  // one elected thread: the pixels of a run that lie inside the row are contiguous in global memory (one bulk copy), the reflected tail of
  // the last run is fetched pixel by pixel (720-byte bulk copies); everything completes on one mbarrier
  auto stage_x = [&](int xs0) {
    if (tid != 0) return;
    const int n = min(kMmaRun, g.Wp - xs0);
    const int nin = max(0, min(n, g.W - xs0));           // pixels of the run inside [0, W)
    fence_proxy_async_smem();                            // the previous run's generic-proxy reads of the buffer precede these async-proxy writes
    mbar_expect_tx(xbar, (uint32_t)(n * kC * 4));
    if (nin > 0) bulk_load(xs_addr, xrow + (long long)xs0 * kC, (uint32_t)(nin * kC * 4), xbar);
    for (int px = nin; px < n; ++px)
      bulk_load(xs_addr + (uint32_t)(px * kC * 4), xrow + (long long)reflect_src(xs0 + px, g.W) * kC, (uint32_t)(kC * 4), xbar);
  };
  auto stage_wait = [&]() { mbar_wait(xbar, xphase); xphase ^= 1u; };
  float gv[3];                                             // 0.5 * channel gates of this image: fetched first, stored after the B fragments
#pragma unroll
  for (int e = 0; e < 3; ++e) {
    const int i = tid + 128 * e, v = i / kCp, c = scc_chan(i - v * kCp);
    gv[e] = c >= 0 ? 0.5f * (v == 0 ? s1 : s2)[(long long)b * kC + c] : 0.f;
  }
  stage_x(0);
  // B fragments of this warp's six n-tiles and the per-column constants
  uint32_t bf[6][2][2][2];
  int cA[6];
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    const int nt = warp * 6 + j;
#pragma unroll
    for (int v = 0; v < 2; ++v)
#pragma unroll
      for (int s = 0; s < 2; ++s)
#pragma unroll
        for (int i = 0; i < 2; ++i) bf[j][v][s][i] = bfrag[((((nt * 2 + v) * 2 + s) * 2 + i) << 5) + lane];
    cA[j] = scc_chan(nt * 8 + tq * 2);                   // an even position is never a pad
  }
#pragma unroll
  for (int e = 0; e < 3; ++e) gs[tid + 128 * e] = gv[e];
  bf16* trow0 = t + ((long long)b * g.Hp + yp) * g.Wp * kCp;
  for (int xs0 = 0; xs0 < g.Wp; xs0 += kMmaRun) {
    const int n = min(kMmaRun, g.Wp - xs0);
    // statistic windows (zero padding of the PADDED map, values gathered through the reflect map)
    for (int i = tid; i < 2 * 3 * (kMmaRun + 2); i += 128) {
      const int v = i / (3 * (kMmaRun + 2)), r2 = i - v * 3 * (kMmaRun + 2);
      const int rr = r2 / (kMmaRun + 2), cc = r2 - rr * (kMmaRun + 2);
      const int yy = yp + rr - 1, xx = xs0 + cc - 1;
      // band mode: row -1 / row Hp of an interior band boundary is the neighbour's statistic row (halo rows of the maps), not zero padding
      const bool inr = yy >= 0 && yy < g.Hp;
      const bool ok = (inr || (yy == -1 && g.top) || (yy == g.Hp && g.bot)) && xx >= 0 && xx < g.Wp;
      const int src = ok ? (inr ? reflect_src(yy, g.H) : (yy < 0 ? -1 : g.H)) * g.W + reflect_src(xx, g.W) : 0;
      sw[i] = ok ? (v == 0 ? ca : cm)[src] : 0.f;
    }
    __syncthreads();                                       // windows written; the previous run's output tile has been copied out
    {                                                      // A rows: thread = (map v, pixel)
      const int v = tid / kMmaRun, px = tid % kMmaRun;
      if (v < 2) {
      const float* wv = sw + v * 3 * (kMmaRun + 2);
      uint16_t hi[9], lo[9];
#pragma unroll
      for (int tap = 0; tap < 9; ++tap) split_bf16(wv[(tap / 3) * (kMmaRun + 2) + px + (tap % 3)], &hi[tap], &lo[tap]);
      uint16_t row[32];
#pragma unroll
      for (int k = 0; k < 32; ++k) row[k] = k < 9 ? hi[k] : k < 18 ? lo[k - 9] : k < 27 ? hi[k - 18] : k < 29 ? (uint16_t)0x3f80 : (uint16_t)0;
      uint4* dst = reinterpret_cast<uint4*>(as + (v * kMmaRun + px) * kMmaAS);
#pragma unroll
      for (int c4 = 0; c4 < 4; ++c4)
        dst[c4] = make_uint4((uint32_t)row[8 * c4] | ((uint32_t)row[8 * c4 + 1] << 16), (uint32_t)row[8 * c4 + 2] | ((uint32_t)row[8 * c4 + 3] << 16),
                             (uint32_t)row[8 * c4 + 4] | ((uint32_t)row[8 * c4 + 5] << 16), (uint32_t)row[8 * c4 + 6] | ((uint32_t)row[8 * c4 + 7] << 16));
      }
    }
    stage_wait();
    __syncthreads();                                       // A rows, gates and this run's token rows are visible
#pragma unroll 1
    for (int pt = 0; pt < kMmaRun / 16; ++pt) {
      if (pt * 16 >= n) break;
      const int r0 = pt * 16 + gq;
      uint32_t af[2][2][4];
#pragma unroll
      for (int v = 0; v < 2; ++v)
#pragma unroll
        for (int s = 0; s < 2; ++s) {
          const uint32_t* a0 = as + (v * kMmaRun + r0) * kMmaAS + s * 8 + tq;
          af[v][s][0] = a0[0]; af[v][s][1] = a0[8 * kMmaAS]; af[v][s][2] = a0[4]; af[v][s][3] = a0[8 * kMmaAS + 4];
        }
      auto mma = [](float* d, const uint32_t* a, uint32_t b0, uint32_t b1) { mma_bf16_16816(d, a[0], a[1], a[2], a[3], b0, b1); };
#pragma unroll
      for (int j = 0; j < 6; ++j) {
        float d1[4] = {0.f, 0.f, 0.f, 0.f}, d2[4] = {0.f, 0.f, 0.f, 0.f};
        mma(d1, af[0][0], bf[j][0][0][0], bf[j][0][0][1]);
        mma(d1, af[0][1], bf[j][0][1][0], bf[j][0][1][1]);
        mma(d2, af[1][0], bf[j][1][0][0], bf[j][1][0][1]);
        mma(d2, af[1][1], bf[j][1][1][0], bf[j][1][1][1]);
        const int pos0 = (warp * 6 + j) * 8 + tq * 2;
        const bool pad = ((pos0 + 1) & 15) == 15;
        const float padv = pos0 < 96 ? 1.0f : 0.f;        // q pads carry the constant 1 (k-gen bias rider), v pads 0
        const float2 g1 = *reinterpret_cast<const float2*>(gs + pos0), g2 = *reinterpret_cast<const float2*>(gs + kCp + pos0);
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const int row = r0 + 8 * hh;
          const float* xr = xs + row * kMmaXS + cA[j];
          const float xa = xr[0], xb = xr[pad ? 0 : 1];
          const float l1a = fmaxf(d1[2 * hh], 0.2f * d1[2 * hh]), l1b = fmaxf(d1[2 * hh + 1], 0.2f * d1[2 * hh + 1]);     // LeakyReLU(0.2) (:329)
          const float l2a = fmaxf(d2[2 * hh], 0.2f * d2[2 * hh]), l2b = fmaxf(d2[2 * hh + 1], 0.2f * d2[2 * hh + 1]);
          const float o0 = fmaf(g2.x, l2a, fmaf(g1.x, l1a, xa));                                                        // (:345-359)
          const float o1 = pad ? padv : fmaf(g2.y, l2b, fmaf(g1.y, l1b, xb));
          os[row * kMmaOS + (pos0 >> 1)] = pack_bf16x2(o0, o1);
        }
      }
    }
    __syncthreads();                                       // output tile complete, token rows consumed
    if (xs0 + kMmaRun < g.Wp) stage_x(xs0 + kMmaRun);     // the next run's rows arrive while this tile is copied out
    bf16* trow = trow0 + (long long)xs0 * kCp;
    if (tid == 32) {                                       // one thread of warp 1 (warp 0's elected thread is busy staging): a bf16 token row leaves as one 384-byte bulk store
      fence_proxy_async_smem();
      const uint32_t os_addr = (uint32_t)__cvta_generic_to_shared(os);
      for (int px = 0; px < n; ++px)
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(trow + (long long)px * kCp), "r"(os_addr + (uint32_t)(px * kMmaOS * 4)), "r"(kCp * 2) : "memory");
      tma_commit();
      tma_wait_read<0>();                                  // the tile may be rewritten after the next barrier
    }
  }
  if (tid == 32) tma_wait_all0();                          // writes complete before the CTA exits
}

// ---------------------------------------------------------------------------------------------
// UnionAttention statistics.  X = a (+ b).
//   rows kernel : CTA per (b, y): channel mean/max per pixel + mean/max over W per channel.
//   cols kernel : CTA per (b, x): mean/max over H per channel.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) ua_rows_kernel(const float* __restrict__ a, const float* __restrict__ bsrc, int B, int H, int W,
                                                      float* __restrict__ cavg, float* __restrict__ cmax, float* __restrict__ wavg, float* __restrict__ wmax) {
  // CTA per (b, y); warp per pixel (lane = channels lane + 32 i), per-channel row statistics carried in registers
  __shared__ float s_sum[8][kCp];
  __shared__ float s_max[8][kCp];
  const int b = blockIdx.x / H, y = blockIdx.x - b * H;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float rs[6], rm[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) { rs[i] = 0.f; rm[i] = -INFINITY; }
  for (int xw = warp; xw < W; xw += 8) {
    const long long off = (((long long)b * H + y) * W + xw) * kC;
    float s = 0.f, m = -INFINITY;
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      const int c = lane + 32 * i;
      if (c < kC) {
        float v = a[off + c];
        if (bsrc != nullptr) v += bsrc[off + c];
        s += v; m = fmaxf(m, v); rs[i] += v; rm[i] = fmaxf(rm[i], v);
      }
    }
    s = warp_sum(s); m = warp_max(m);
    if (lane == 0) { cavg[((long long)b * H + y) * W + xw] = s / (float)kC; cmax[((long long)b * H + y) * W + xw] = m; }
  }
#pragma unroll
  for (int i = 0; i < 6; ++i) { s_sum[warp][lane + 32 * i] = rs[i]; s_max[warp][lane + 32 * i] = rm[i]; }
  __syncthreads();
  const int c = threadIdx.x;
  if (c < kC) {
    float s = 0.f, m = -INFINITY;
#pragma unroll
    for (int wv = 0; wv < 8; ++wv) { s += s_sum[wv][c]; m = fmaxf(m, s_max[wv][c]); }
    wavg[((long long)b * H + y) * kC + c] = s / (float)W;
    wmax[((long long)b * H + y) * kC + c] = m;
  }
}

__global__ void __launch_bounds__(192) ua_cols_kernel(const float* __restrict__ a, const float* __restrict__ bsrc, int B, int H, int W,
                                                      float* __restrict__ havg, float* __restrict__ hmax, int Hf) {
  const int b = blockIdx.x / W, xw = blockIdx.x - b * W;
  const int c = threadIdx.x;
  if (c >= kC) return;
  float s = 0.f, m = -INFINITY;
  for (int y = 0; y < H; ++y) {
    const long long off = (((long long)b * H + y) * W + xw) * kC + c;
    float v = a[off]; if (bsrc != nullptr) v += bsrc[off];
    s += v; m = fmaxf(m, v);
  }
  havg[((long long)b * kC + c) * W + xw] = s / (float)Hf;       // band mode: this band's share of the frame mean (all-reduced by SUM)
  hmax[((long long)b * kC + c) * W + xw] = m;
}

// 3x3 conv 2->1 on a (rows x cols) plane pair, zero padded.  plane layouts: avg/max [B][rows][cols]
// top / bot: row -1 / row `rows` exists (halo row of the neighbour band); tr: the filter is applied transposed (plane stored [cols][rows] ...)
__device__ __forceinline__ float conv2to1(const float* __restrict__ pa, const float* __restrict__ pm, int rows, int cols, int rr, int cc,
                                          const float* __restrict__ w, float bias, int top = 0, int bot = 0, bool tr = false) {
  float acc = bias;
#pragma unroll
  for (int ky = 0; ky < 3; ++ky) {
    const int r2 = rr + ky - 1;
    if ((r2 < 0 && !(top && r2 == -1)) || (r2 >= rows && !(bot && r2 == rows))) continue;
#pragma unroll
    for (int kx = 0; kx < 3; ++kx) {
      const int c2 = cc + kx - 1;
      if (c2 < 0 || c2 >= cols) continue;
      const int wi = tr ? kx * 3 + ky : ky * 3 + kx;
      acc += w[wi] * pa[(long long)r2 * cols + c2] + w[9 + wi] * pm[(long long)r2 * cols + c2];
    }
  }
  return acc;
}

__global__ void ua_small_convs_kernel(int B, int H, int W, UaW w, const float* __restrict__ cavg, const float* __restrict__ cmax,
                                      const float* __restrict__ havg, const float* __restrict__ hmax, const float* __restrict__ wavg,
                                      const float* __restrict__ wmax, float* __restrict__ c_att, float* __restrict__ h_att, float* __restrict__ w_att,
                                      int top, int bot) {
  const long long n1 = (long long)B * H * W, n2 = (long long)B * kC * W, n3 = (long long)B * kC * H;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < n1 + n2 + n3; idx += (long long)gridDim.x * blockDim.x) {
    if (idx < n1) {                 // conv1 over the (H, W) plane                       (:120-122)
      const int b = (int)(idx / (H * W)); const int rem = (int)(idx - (long long)b * H * W);
      c_att[idx] = conv2to1(cavg + (long long)b * H * W, cmax + (long long)b * H * W, H, W, rem / W, rem % W, w.c1_w, w.c1_b[0], top, bot);
    } else if (idx < n1 + n2) {     // conv2 over the (channel, W) plane                 (:124-126)
      const long long i = idx - n1;
      const int b = (int)(i / (kC * W)); const int rem = (int)(i - (long long)b * kC * W);
      h_att[((long long)b * W + rem % W) * kC + rem / W] =      // stored [b][x][c] (channel fastest) for ua_build
          conv2to1(havg + (long long)b * kC * W, hmax + (long long)b * kC * W, kC, W, rem / W, rem % W, w.c2_w, w.c2_b[0]);
    } else {                        // conv3 over the (channel, H) plane                 (:128-130); the plane is stored [y][c], filter transposed
      const long long i = idx - n1 - n2;
      const int b = (int)(i / (kC * H)); const int rem = (int)(i - (long long)b * kC * H);
      w_att[(long long)b * H * kC + rem] =                      // stored [b][y][c]
          conv2to1(wavg + (long long)b * kC * H, wmax + (long long)b * kC * H, H, kC, rem / kC, rem % kC, w.c3_w, w.c3_b[0], top, bot, true);
    }
  }
}

// thread = (pixel, 8 channels); h_att [b][x][c], w_att [b][y][c]
__global__ void ua_build_kernel(int B, int H, int W, const float* __restrict__ c_att, const float* __restrict__ h_att, const float* __restrict__ w_att,
                                bf16* __restrict__ s) {
  constexpr int groups = kCp / 8;
  const long long total = (long long)B * H * W * groups;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int gi = (int)(idx % groups);
    const long long pix = idx / groups;
    const int xw = (int)(pix % W); const long long t = pix / W; const int y = (int)(t % H); const int b = (int)(t / H);
    const int c0 = gi * 8;
    float v[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) v[e] = 0.f;
    if (c0 < kC) {
      const float ca = c_att[pix];
      const float* wa = w_att + ((long long)b * H + y) * kC + c0;
      const float* ha = h_att + ((long long)b * W + xw) * kC + c0;
      const float4 w0 = *reinterpret_cast<const float4*>(wa), h0 = *reinterpret_cast<const float4*>(ha);
      v[0] = ca + w0.x + h0.x; v[1] = ca + w0.y + h0.y; v[2] = ca + w0.z + h0.z; v[3] = ca + w0.w + h0.w;      // (:133)
      if (c0 + 4 < kC) {
        const float4 w1 = *reinterpret_cast<const float4*>(wa + 4), h1 = *reinterpret_cast<const float4*>(ha + 4);
        v[4] = ca + w1.x + h1.x; v[5] = ca + w1.y + h1.y; v[6] = ca + w1.z + h1.z; v[7] = ca + w1.w + h1.w;
      }
    }
    *reinterpret_cast<uint4*>(s + pix * kCp + c0) =
        make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
  }
}

// thread = (pixel, 4 consecutive channels): 180 = 45 chunks of 4, chunks 45..47 are the zero pad of the bf16 operand row.  sigmoid(x) =
// 0.5 + 0.5 tanh(x / 2) on one MUFU op (tanh.approx.f32: relative error <= 2^-10.987, so <= 2^-11.987 absolute here); the element-per-thread
// version with three exp + divide sigmoids and a 64-bit division per element was instruction-bound at 3.2 TB/s.
__device__ __forceinline__ float sigmoid_fast(float x) { return fmaf(0.5f, tanh_approx(0.5f * x), 0.5f); }
__global__ void __launch_bounds__(256) fusion_combine_kernel(const float* __restrict__ first, const float* __restrict__ second, const float* __restrict__ a1,
                                                             const float* __restrict__ a2, const float* __restrict__ a3, bf16* __restrict__ out,
                                                             float* __restrict__ of, long long N) {
  constexpr int kChunks = kCp / 4;   // 48
  const long long total = N * kChunks;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const long long r = idx / kChunks; const int c4 = (int)(idx - r * kChunks);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c4 < kC / 4) {
      const long long i = r * kC + 4 * c4;
      const float4 f = *reinterpret_cast<const float4*>(first + i), sc = *reinterpret_cast<const float4*>(second + i);
      const float4 x1 = *reinterpret_cast<const float4*>(a1 + i), x2 = *reinterpret_cast<const float4*>(a2 + i), x3 = *reinterpret_cast<const float4*>(a3 + i);
      const float t0 = sigmoid_fast(x2.x), t1 = sigmoid_fast(x2.y), t2 = sigmoid_fast(x2.z), t3 = sigmoid_fast(x2.w);                  // (:152)
      v.x = f.x * sigmoid_fast(x1.x * t0) + sc.x * sigmoid_fast(x3.x * (1.f - t0));                                                  // (:155-162)
      v.y = f.y * sigmoid_fast(x1.y * t1) + sc.y * sigmoid_fast(x3.y * (1.f - t1));
      v.z = f.z * sigmoid_fast(x1.z * t2) + sc.z * sigmoid_fast(x3.z * (1.f - t2));
      v.w = f.w * sigmoid_fast(x1.w * t3) + sc.w * sigmoid_fast(x3.w * (1.f - t3));
      if (of != nullptr) *reinterpret_cast<float4*>(of + i) = v;
    }
    *reinterpret_cast<uint2*>(out + r * kCp + 4 * c4) = make_uint2(pack_bf16x2(v.x, v.y), pack_bf16x2(v.z, v.w));
  }
}

inline int grid_for(long long total, int block) {
  long long g = (total + block - 1) / block;
  const long long cap = 148LL * 16;
  return (int)(g < cap ? (g > 0 ? g : 1) : cap);
}

}  // namespace

int launch_entry_im2col(const float* x, bf16* a0, int B, int H, int W, int in_ch, int f, int Kp, const float* mean3, float img_range, cudaStream_t st,
                        int y0, int Hf) {
  if (in_ch > 3 || f > 9 || Kp > 512 || Kp % 8 != 0) { set_error("launch_entry_im2col: footprint %d x %d x %d / Kp %d not supported", f, f, in_ch, Kp); return 1; }
  const int nseg = (W + kImSeg - 1) / kImSeg;
  const long long ctas = (long long)B * H * nseg;
  if (ctas > 2147483647LL) { set_error("launch_entry_im2col: too many rows"); return 1; }
  entry_im2col_kernel<<<(unsigned)ctas, 256, 0, st>>>(x, a0, B, H, W, in_ch, f, Kp, mean3[0], mean3[1], mean3[2], img_range, nseg, y0, Hf > 0 ? Hf : H);
  HITSIR_CHECK(cudaGetLastError());
  return 0;
}
int launch_ln_rows(const float* x, const float* gamma, const float* beta, bf16* ob, float* of, long long N, cudaStream_t st, const float* add,
                   long long add_rows) {
  ln_rows_kernel<<<grid_for(N * 32, 256), 256, 0, st>>>(x, gamma, beta, ob, of, N, add, add_rows > 0 ? add_rows : 1);
  HITSIR_CHECK(cudaGetLastError());
  return 0;
}
int launch_u8hwc_to_f32nchw(const uint8_t* in, float* out, int B, int H, int W, int C, cudaStream_t st) {
  u8hwc_to_f32nchw_kernel<<<grid_for((long long)B * C * H * W, 256), 256, 0, st>>>(in, out, B, H, W, C);
  HITSIR_CHECK(cudaGetLastError());
  return 0;
}
int launch_f32nchw_to_u8hwc(const float* in, uint8_t* out, int B, int H, int W, int C, cudaStream_t st) {
  f32nchw_to_u8hwc_kernel<false><<<grid_for((long long)B * C * H * W, 256), 256, 0, st>>>(in, out, B, H, W, C);
  HITSIR_CHECK(cudaGetLastError());
  return 0;
}
int launch_f32nchw_to_u8hwc_round(const float* in, uint8_t* out, int B, int H, int W, int C, cudaStream_t st) {
  f32nchw_to_u8hwc_kernel<true><<<grid_for((long long)B * C * H * W, 256), 256, 0, st>>>(in, out, B, H, W, C);
  HITSIR_CHECK(cudaGetLastError());
  return 0;
}
int launch_f32_to_f32_tap(const void* src, int is_bf16, int ld, float* dst, long long rows, int cols, int perm, cudaStream_t st) {
  tap_kernel<<<grid_for(rows * cols, 256), 256, 0, st>>>(src, is_bf16, ld, dst, rows, cols, perm);
  HITSIR_CHECK(cudaGetLastError());
  return 0;
}
int launch_cast_rows_bf16(const float* a, bf16* out, long long N, cudaStream_t st) {
  cast_rows_bf16_kernel<<<grid_for(N * (kCp / 8), 256), 256, 0, st>>>(a, out, N);
  HITSIR_CHECK(cudaGetLastError());
  return 0;
}
int launch_add_to_bf16(const float* a, const float* b, bf16* out, long long N, cudaStream_t st) {
  add_to_bf16_kernel<<<grid_for(N * kCp, 256), 256, 0, st>>>(a, b, out, N);
  HITSIR_CHECK(cudaGetLastError());
  return 0;
}
int launch_sca_stats(const float* x, PadGeom g, float* cavg, float* cmax, float* part_sum, float* part_max, int nparts, cudaStream_t st) {
  dim3 grid(nparts, g.B);
  sca_stats_kernel<<<grid, 256, 0, st>>>(x, g, cavg, cmax, part_sum, part_max, nparts);
  HITSIR_CHECK(cudaGetLastError());
  return 0;
}
__global__ void reduce_parts_kernel(const float* __restrict__ part_sum, const float* __restrict__ part_max, int nparts, float* __restrict__ out_sum,
                                    float* __restrict__ out_max) {
  const int c = threadIdx.x;
  if (c >= kC) return;
  // same association as sca_mlp_kernel (four strided groups merged in order), so that a frame run as ONE band reproduces the ordinary forward bit for bit
  float s[4] = {0.f, 0.f, 0.f, 0.f}, m = -INFINITY;
#pragma unroll
  for (int g = 0; g < 4; ++g)
    for (int p = g; p < nparts; p += 4) { s[g] += part_sum[(long long)p * kC + c]; m = fmaxf(m, part_max[(long long)p * kC + c]); }
  out_sum[c] = ((s[0] + s[1]) + s[2]) + s[3]; out_max[c] = m;
}
int launch_reduce_parts(const float* part_sum, const float* part_max, int nparts, float* out_sum, float* out_max, cudaStream_t st) {
  reduce_parts_kernel<<<1, 192, 0, st>>>(part_sum, part_max, nparts, out_sum, out_max);
  HITSIR_CHECK(cudaGetLastError());
  return 0;
}
int launch_sca_mlp(const float* part_sum, const float* part_max, int nparts, PadGeom g, CasaW w, float* s1, float* s2, cudaStream_t st) {
  HITSIR_CHECK(launch_pdl(sca_mlp_kernel, dim3(g.B), dim3(768), 0, st, part_sum, part_max, nparts, g, w, s1, s2));
  return 0;
}
int launch_qkv_build(const float* x, PadGeom g, int casa, const float* cavg, const float* cmax, const float* s1, const float* s2, CasaW w, bf16* t,
                     cudaStream_t st) {
  if (casa) {
    if (w.bfrag == nullptr) { set_error("launch_qkv_build: casa B fragments were not packed"); return 1; }
    static unsigned long long configured = 0;
    if (ensure_dynamic_smem(qkv_casa_mma_kernel, kMmaSmem, &configured)) return 1;
    HITSIR_CHECK(launch_pdl(qkv_casa_mma_kernel, dim3(g.B * g.Hp), dim3(128), kMmaSmem, st, x, g, cavg, cmax, s1, s2, w.bfrag, t));
    return 0;
  }
  const long long total = (long long)g.B * g.Hp * g.Wp * (kCp / 8);
  qkv_build_kernel<<<grid_for(total, 192), 192, 0, st>>>(x, g, t);
  HITSIR_CHECK(cudaGetLastError());
  return 0;
}
int casa_bfrag_words() { return kCasaBfragWords; }
int launch_pack_casa_bfrag(CasaW w, uint32_t* img, cudaStream_t st) {
  casa_bfrag_kernel<<<(kCasaBfragWords + 255) / 256, 256, 0, st>>>(w, img);
  HITSIR_CHECK(cudaGetLastError());
  return 0;
}
int launch_ua_stats(const float* a, const float* b, int B, int H, int W, float* cavg, float* cmax, float* havg, float* hmax, float* wavg, float* wmax,
                    cudaStream_t st, int Hf) {
  ua_rows_kernel<<<B * H, 256, 0, st>>>(a, b, B, H, W, cavg, cmax, wavg, wmax);
  HITSIR_CHECK(cudaGetLastError());
  ua_cols_kernel<<<B * W, 192, 0, st>>>(a, b, B, H, W, havg, hmax, Hf > 0 ? Hf : H);
  HITSIR_CHECK(cudaGetLastError());
  return 0;
}
int launch_ua_small_convs(int B, int H, int W, UaW w, const float* cavg, const float* cmax, const float* havg, const float* hmax, const float* wavg,
                          const float* wmax, float* c_att, float* h_att, float* w_att, cudaStream_t st, int top, int bot) {
  const long long total = (long long)B * H * W + (long long)B * kC * W + (long long)B * kC * H;
  ua_small_convs_kernel<<<grid_for(total, 256), 256, 0, st>>>(B, H, W, w, cavg, cmax, havg, hmax, wavg, wmax, c_att, h_att, w_att, top, bot);
  HITSIR_CHECK(cudaGetLastError());
  return 0;
}
int launch_ua_build(int B, int H, int W, const float* c_att, const float* h_att, const float* w_att, bf16* s, cudaStream_t st) {
  const long long total = (long long)B * H * W * (kCp / 8);
  ua_build_kernel<<<grid_for(total, 256), 256, 0, st>>>(B, H, W, c_att, h_att, w_att, s);
  HITSIR_CHECK(cudaGetLastError());
  return 0;
}
int launch_fusion_combine(const float* first, const float* second, const float* a1, const float* a2, const float* a3, bf16* out, float* of, long long N,
                          cudaStream_t st) {
  fusion_combine_kernel<<<grid_for(N * (kCp / 4), 256), 256, 0, st>>>(first, second, a1, a2, a3, out, of, N);
  HITSIR_CHECK(cudaGetLastError());
  return 0;
}

}  // namespace hitsir
