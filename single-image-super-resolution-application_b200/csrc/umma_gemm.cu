// tcgen05 / TMEM / TMA dense-contraction kernel for sm_100a.
//
// Persistent, warp-specialised:  warp 0 = TMA producer (one lane), warp 1 = tcgen05.mma issuer
// (one lane), warp 2 = TMEM allocator, warps 4..7 = epilogue (thread r <-> accumulator row r,
// TMEM lane r).  Operands are staged by TMA into 128B-swizzled K-major shared-memory tiles
// (A: 128 rows x 64 bf16, B: BN rows x 64 bf16 per stage), the fp32 accumulator tile
// (128 x BN) lives in TMEM and is double-buffered so the epilogue of tile i overlaps the MMAs
// of tile i+1.  The mainloop serves token-major linears (2-D tensor map) and 3x3 convolutions
// as implicit GEMM (4-D NHWC tensor map, one TMA box per filter tap, zero padding from TMA
// out-of-bounds fill); the epilogue stores each row's values straight to global memory, which
// is what the pixel-shuffle heads (EPI_SHUFFLE_*, gemm.cuh) need.  Every other epilogue runs on
// the TMA-staged kernel (umma_gemm_tma.cu).
#include "gemm.cuh"

namespace hitsir {

template <int BN>
struct UmmaCfg {
  static constexpr int kStages = (BN >= 192) ? 4 : 6;
  static constexpr int kABytes = 128 * 128;          // 128 rows x 64 bf16
  static constexpr int kBBytes = BN * 128;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kTmemCols = (2 * BN <= 32) ? 32 : (2 * BN <= 64) ? 64 : (2 * BN <= 128) ? 128 : (2 * BN <= 256) ? 256 : 512;
  static constexpr int kSmemBytes = kStages * kStageBytes + 1024 /*align slack*/ + 256 /*barriers*/;
};

struct TmemAcc {
  uint32_t base;   // lane + column base of this thread's row in the current accumulator stage
  __device__ __forceinline__ void load16(int c0, float* v) {
    __syncwarp();   // tcgen05.ld is .sync.aligned: reconverge after per-row predicated stores
    tmem_ld16(base + (uint32_t)c0, v);
  }
};

template <int BN>
__global__ void __launch_bounds__(256, 1)
umma_gemm_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b, const GemmParams p) {
  using Cfg = UmmaCfg<BN>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_al = smem_raw + (smem_base - smem_u32(smem_raw));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_al + Cfg::kStages * Cfg::kStageBytes);
  // barrier map: [0,S) full, [S,2S) empty, [2S,2S+2) tmem_full, [2S+2,2S+4) tmem_empty, then tmem ptr
  const uint32_t bar0 = smem_u32(bars);
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (Cfg::kStages + s); };
  auto tfull_bar = [&](int s) { return bar0 + 8u * (2 * Cfg::kStages + s); };
  auto tempty_bar = [&](int s) { return bar0 + 8u * (2 * Cfg::kStages + 2 + s); };
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 2 * Cfg::kStages + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int total = p.m_tiles * p.n_tiles;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < Cfg::kStages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(tfull_bar(s), 1); mbar_init(tempty_bar(s), 128); }
    fence_barrier_init();
  }
  if (warp == 2) {
    tmem_alloc(smem_u32(tmem_ptr_smem), Cfg::kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    if (lane == 0) {
      // ===================== TMA producer =====================
      int stage = 0; uint32_t phase = 0;
      for (int w = blockIdx.x; w < total; w += gridDim.x) {
        const int n_tile = w % p.n_tiles, m_tile = w / p.n_tiles;
        const ConvTile t = p.conv ? conv_tile(m_tile, p.tiles_x, p.tiles_y) : ConvTile{0, 0, 0};
        for (int kb = 0; kb < p.num_kb; ++kb) {
          mbar_wait(empty_bar(stage), phase ^ 1u);
          const uint32_t sa = smem_base + stage * Cfg::kStageBytes;
          const uint32_t sb = sa + Cfg::kABytes;
          mbar_expect_tx(full_bar(stage), Cfg::kStageBytes);
          if (p.conv) {
            const int tap = kb / p.cblocks, cb = kb - tap * p.cblocks;
            const int dy = tap / 3 - 1, dx = tap % 3 - 1;
            tma_load_4d(sa, &tmap_a, full_bar(stage), cb * 64, t.x0 + dx, t.y0 + dy + p.a_y_off, t.b);
          } else {
            tma_load_2d(sa, &tmap_a, full_bar(stage), kb * 64, m_tile * 128);
          }
          tma_load_2d(sb, &tmap_b, full_bar(stage), kb * 64, n_tile * BN);
          if (++stage == Cfg::kStages) { stage = 0; phase ^= 1u; }
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
        const uint32_t aphase = (uint32_t)(it >> 1) & 1u;
        mbar_wait(tempty_bar(as), aphase ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(as * BN);
        for (int kb = 0; kb < p.num_kb; ++kb) {
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          const uint32_t sa = smem_base + stage * Cfg::kStageBytes;
          const uint32_t sb = sa + Cfg::kABytes;
          const uint64_t adesc = umma_desc_sw128(sa);
          const uint64_t bdesc = umma_desc_sw128(sb);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            // advance 16 bf16 = 32 B along K inside the 128B swizzle atom: +2 in the (addr>>4) field
            umma_bf16(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (kb | k) != 0 ? 1u : 0u);
          }
          umma_commit(empty_bar(stage));          // frees the smem stage when these MMAs retire
          if (++stage == Cfg::kStages) { stage = 0; phase ^= 1u; }
        }
        umma_commit(tfull_bar(as));               // accumulator tile complete -> epilogue
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue =====================
    const int ew = warp & 3;                      // TMEM lane quarter this warp may access
    const int r = ew * 32 + lane;
    int it = 0;
    for (int w = blockIdx.x; w < total; w += gridDim.x, ++it) {
      const int n_tile = w % p.n_tiles, m_tile = w / p.n_tiles;
      const int as = it & 1;
      const uint32_t aphase = (uint32_t)(it >> 1) & 1u;
      mbar_wait(tfull_bar(as), aphase);
      tc_fence_after();
      TmemAcc acc;
      acc.base = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(as * BN);
      const RowInfo ri = row_info(p, m_tile, r);
      epilogue_row<BN>(p, acc, ri, n_tile);
      tc_fence_before();
      mbar_arrive(tempty_bar(as));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// Every tensor map of the library: a `rank`-D (2 or 4) tensor of fp32 (elem_bytes 4) or bf16 elements, dims and box innermost first,
// `strides` the rank - 1 outer strides in bytes; boxes land in 128B-swizzled shared memory, out-of-bounds elements read as zero.
static int encode_tmap(CUtensorMap* m, const void* base, int elem_bytes, int rank, const cuuint64_t* dims, const cuuint64_t* strides,
                       const cuuint32_t* box) {
  static PFN_encodeTiled enc = nullptr;
  if (enc == nullptr) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || ptr == nullptr) {
      set_error("cudaGetDriverEntryPoint(cuTensorMapEncodeTiled) failed: %s", cudaGetErrorString(e));
      return 1;
    }
    enc = reinterpret_cast<PFN_encodeTiled>(ptr);
  }
  const cuuint32_t es[4] = {1, 1, 1, 1};
  const CUresult r = enc(m, elem_bytes == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank,
                         const_cast<void*>(base), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char shape[320];
    int n = snprintf(shape, sizeof(shape), "%d-byte elements, dims", elem_bytes);
    for (int i = 0; i < rank; ++i) n += snprintf(shape + n, sizeof(shape) - n, " %llu", (unsigned long long)dims[i]);
    n += snprintf(shape + n, sizeof(shape) - n, ", byte strides");
    for (int i = 0; i < rank - 1; ++i) n += snprintf(shape + n, sizeof(shape) - n, " %llu", (unsigned long long)strides[i]);
    n += snprintf(shape + n, sizeof(shape) - n, ", box");
    for (int i = 0; i < rank; ++i) n += snprintf(shape + n, sizeof(shape) - n, " %u", box[i]);
    set_error("cuTensorMapEncodeTiled(%s) failed with CUresult %d", shape, (int)r);
    return 1;
  }
  return 0;
}

int make_tmap_2d(CUtensorMap* m, const void* base, uint64_t inner, uint64_t outer, uint64_t pitch_bytes,
                 uint32_t box_inner, uint32_t box_outer) {
  return make_tmap_2d_t(m, base, 2, inner, outer, pitch_bytes, box_inner, box_outer);
}

int make_tmap_2d_t(CUtensorMap* m, const void* base, int elem_bytes, uint64_t inner, uint64_t outer, uint64_t pitch_bytes,
                   uint32_t box_inner, uint32_t box_outer) {
  const cuuint64_t dims[2] = {inner, outer}, strides[1] = {pitch_bytes};
  const cuuint32_t box[2] = {box_inner, box_outer};
  return encode_tmap(m, base, elem_bytes, 2, dims, strides, box);
}

int make_tmap_nhwc(CUtensorMap* m, const void* base, int B, int H, int W, int Cpad, uint32_t box_c, uint32_t box_w, uint32_t box_h) {
  return make_tmap_nhwc_t(m, base, 2, B, H, W, Cpad, Cpad, box_c, box_w, box_h);
}

// NHWC tensor with `C` visible channels out of a pixel pitch of `ldc` elements
int make_tmap_nhwc_t(CUtensorMap* m, const void* base, int elem_bytes, int B, int H, int W, int C, int ldc, uint32_t box_c, uint32_t box_w,
                     uint32_t box_h) {
  const cuuint64_t pix = (cuuint64_t)ldc * elem_bytes;
  const cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B}, strides[3] = {pix, W * pix, (cuuint64_t)H * W * pix};
  const cuuint32_t box[4] = {box_c, box_w, box_h, 1};
  return encode_tmap(m, base, elem_bytes, 4, dims, strides, box);
}

int make_tmap_nhwc_strided(CUtensorMap* m, const void* base, int B, int H, int W, int C, uint64_t pix_bytes, uint64_t row_bytes, uint64_t img_bytes,
                           uint32_t box_c, uint32_t box_w, uint32_t box_h) {
  const cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B}, strides[3] = {pix_bytes, row_bytes, img_bytes};
  const cuuint32_t box[4] = {box_c, box_w, box_h, 1};
  return encode_tmap(m, base, 2, 4, dims, strides, box);
}

template <int BN>
static int launch_bn(const GemmParams& p, const CUtensorMap& ta, const CUtensorMap& tb, int num_sms, cudaStream_t st) {
  using Cfg = UmmaCfg<BN>;
  static unsigned long long configured = 0;
  if (ensure_dynamic_smem(umma_gemm_kernel<BN>, Cfg::kSmemBytes, &configured)) return 1;
  const int total = p.m_tiles * p.n_tiles;
  const int grid = total < num_sms ? total : num_sms;
  if (grid <= 0) return 0;
  umma_gemm_kernel<BN><<<grid, 256, Cfg::kSmemBytes, st>>>(ta, tb, p);
  HITSIR_CHECK(cudaGetLastError());
  return 0;
}

int launch_umma_gemm(int BN, const GemmParams& p, const CUtensorMap& ta, const CUtensorMap& tb, int num_sms, cudaStream_t st) {
  if (p.epi != EPI_SHUFFLE_NCHW && p.epi != EPI_SHUFFLE_BF16) { set_error("launch_umma_gemm: epilogue %d is not a pixel shuffle", p.epi); return 1; }
  switch (BN) {
    case 16: return launch_bn<16>(p, ta, tb, num_sms, st);
    case 32: return launch_bn<32>(p, ta, tb, num_sms, st);
    case 64: return launch_bn<64>(p, ta, tb, num_sms, st);
    case 192: return launch_bn<192>(p, ta, tb, num_sms, st);
    case 256: return launch_bn<256>(p, ta, tb, num_sms, st);
    default: set_error("launch_umma_gemm: unsupported N tile %d", BN); return 1;
  }
}

}  // namespace hitsir
