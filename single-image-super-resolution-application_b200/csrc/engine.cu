// hitsir_b200 engine: parameter registry (reference state_dict keys), weight packing, workspace
// layout and the forward-pass orchestration of HiT_SIR.forward
// (/root/reference/models/hit_sir_pro.py:1304-1344) behind the C ABI of include/hitsir_b200.h.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <string>
#include <vector>

#include "../../include/hitsir_b200.h"
#include "gemm.cuh"
#include "kernels.cuh"

namespace hitsir {

static thread_local char g_err[2048] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

struct ParamSpec {
  std::string name;
  int64_t numel;
  size_t offset;   // floats into the master arena
  bool set;
};

// one packed dense operand (bf16 [Npad][K]) + fp32 bias [Npad] + its TMA descriptor
struct GemmW {
  bf16* w = nullptr;
  float* b = nullptr;
  int Npad = 0, K = 0, BN = 0;
  CUtensorMap tm;
  bf16* wf = nullptr;          // conv_last 64 -> in_chans only: the nine taps folded into N, [48][64] (launch_conv_last_fold)
  CUtensorMap tmf;
};

struct BlockW {
  int win = 0, base = 0, r = 0;
  const float *g1, *b1, *g2, *b2;
  CasaW casa;
  float *casa_w1 = nullptr, *casa_w2 = nullptr;
  uint32_t* casa_bfrag = nullptr;
  SccW scc;
  float* bias_tbl = nullptr;
  uint8_t *pool_img = nullptr, *bias_img = nullptr, *w_img = nullptr;
  GemmW proj, fc1, fc2;
  float *dw_w = nullptr, *dw_b = nullptr;
  uint32_t* dw_mma = nullptr;
  uint8_t* w2_img = nullptr;
};

struct UaPack {
  UaW small;
  GemmW conv_last;
};

// optional per-category CUDA-event timing of the launches of a forward (bench.py's live roofline numbers)
struct ProfRec { int cat; cudaEvent_t a, b; };
struct Prof {
  bool on = false;
  std::vector<std::string> cats;
  std::vector<ProfRec> recs;
  std::vector<cudaEvent_t> pool;   // recycled events
  int cat_id(const char* name) {
    for (size_t i = 0; i < cats.size(); ++i) if (cats[i] == name) return (int)i;
    cats.push_back(name);
    return (int)cats.size() - 1;
  }
  cudaEvent_t get() {
    if (!pool.empty()) { cudaEvent_t e = pool.back(); pool.pop_back(); return e; }
    cudaEvent_t e; cudaEventCreate(&e); return e;
  }
};

struct Tap {
  std::string name;
  float* dst = nullptr;
  int64_t floats = 0;
  int stop = 0;
};

// test hook: replaces a named activation with caller data before it is consumed (a forward *pre*-hook that returns a new input)
struct Inject {
  std::string name;
  const float* src = nullptr;
  int64_t floats = 0;
};

}  // namespace hitsir

using namespace hitsir;

struct HitsirHandle {
  HitsirConfig cfg;
  int device = 0;
  int num_sms = 148;
  // A/B switches: only a test build (-DHITSIR_AB_PATHS, build.py --ab) can turn them on; the product has ONE path and they stay false
  bool simt = false;
  bool projfc1_fused = false;     // HITSIR_PROJFC1=fused: proj + fc1 chained in one kernel (proj_fc1.cu; slower than the two GEMM launches so far, DESIGN.md 3.7)
  bool b_streamed = false;        // HITSIR_GEMMW=streamed: linears re-load their weight tile per 128-token tile (A/B switch)
  bool no_epilogue_stats = false; // HITSIR_STATS=kernel: always compute the casa statistics with the stand-alone sca_stats pass
  bool ffn_unfused = false;       // HITSIR_FFN=unfused: separate dwconv5 and fc2 kernels for every block
  bool scc_gram_only = false;     // HITSIR_SCC=gram: use the Gram-matrix kernel (scc_umma.cu) for every window size
  bool direct_epilogue = false;   // HITSIR_EPILOGUE=direct: per-row global stores instead of the TMA-staged epilogue
  std::vector<ParamSpec> params;
  std::map<std::string, int> index;
  float* arena = nullptr;      // device fp32 master copy of every parameter
  size_t arena_floats = 0;
  bool finalized = false;
  // packed buffers live in a few large chunks (bump-allocated in a fixed order, so a re-pack after a weight update lands every table at the
  // same address): ~600 cudaMalloc / cudaFree pairs per hitsir_finalize_weights were most of its 60-140 ms
  std::vector<void*> owned;    // chunks
  std::vector<size_t> chunk_bytes;
  size_t chunk_cur = 0, chunk_off = 0;
  // packed weights
  GemmW first, first_last;     // conv_first (im2col GEMM) and its 1x1 conv_last (ms only)
  int first_f = 3, first_kp = 64;
  std::vector<std::vector<BlockW>> blocks;
  std::vector<GemmW> layer_conv;
  GemmW conv_after_body;
  // resi_connection='3conv': [C -> C/4 3x3] LeakyReLU [C/4 -> C/4 1x1] LeakyReLU [C/4 -> C 3x3]; index num_layers = conv_after_body
  std::vector<GemmW> r3_a, r3_b, r3_c;
  UaPack ua[3];
  GemmW conv_before_upsample, conv_up1, conv_up2, conv_hr, conv_last;
  std::vector<GemmW> upsample;   // pixelshuffle stages / pixelshuffledirect
  float mean[4] = {0, 0, 0, 0};
  // per-forward state
  Tap tap;
  Inject inject;
  int64_t launches = 0;
  Prof prof;
};

namespace {

const int kNumFeat = 64;

int win_of(const HitsirConfig& c, int j) { return (int)(c.base_win_size[0] * c.hier_win_ratios[j]); }

void add_param(HitsirHandle* h, const std::string& name, int64_t numel) {
  ParamSpec p{name, numel, h->arena_floats, false};
  h->arena_floats += (size_t)((numel + 3) / 4 * 4);   // keep every tensor 16-byte aligned
  h->index[name] = (int)h->params.size();
  h->params.push_back(p);
}
void add_wb(HitsirHandle* h, const std::string& prefix, int64_t wn, int64_t bn) {
  add_param(h, prefix + ".weight", wn);
  add_param(h, prefix + ".bias", bn);
}

void build_param_list(HitsirHandle* h) {
  const HitsirConfig& c = h->cfg;
  const int C = c.embed_dim, ic = c.in_chans;
  if (c.is_mult_size_conv_feat_extract) {
    add_wb(h, "conv_first.conv3", (int64_t)C * ic * 9, C);
    add_wb(h, "conv_first.conv5", (int64_t)C * ic * 25, C);
    add_wb(h, "conv_first.conv7", (int64_t)C * ic * 49, C);
    add_wb(h, "conv_first.conv9", (int64_t)C * ic * 81, C);
    add_wb(h, "conv_first.conv_x", (int64_t)C * 3, C);          // nn.Conv2d(3, ...) hard-coded (:59)
    add_wb(h, "conv_first.norm", C, C);                         // registered but never applied (:62)
    add_wb(h, "conv_first.conv_last", (int64_t)C * 4 * C, C);
  } else {
    add_wb(h, "conv_first", (int64_t)C * ic * 9, C);
  }
  if (c.is_fusion) {
    for (int u = 1; u <= 3; ++u) {
      const std::string p = "fusion.union_attention" + std::to_string(u);
      add_wb(h, p + ".conv1", 18, 1);
      add_wb(h, p + ".conv2", 18, 1);
      add_wb(h, p + ".conv3", 18, 1);
      add_wb(h, p + ".conv_last", (int64_t)C * C * 9, C);
    }
  }
  if (c.ape_tokens > 0) add_param(h, "absolute_pos_embed", (int64_t)c.ape_tokens * C);
  add_wb(h, "patch_embed.norm", C, C);
  const int hd = C / (2 * c.num_heads[0]);
  const int pos_dim = (C / 4) / 4;
  const int hidden = (int)(C * c.mlp_ratio);
  for (int i = 0; i < c.num_layers; ++i) {
    for (int j = 0; j < c.depths[i]; ++j) {
      const std::string p = "layers." + std::to_string(i) + ".residual_group.blocks." + std::to_string(j);
      const int w = win_of(c, j), base = w < c.base_win_size[0] ? w : c.base_win_size[0], r = w / base;
      add_wb(h, p + ".norm1", C, C);
      if (c.is_channel_spatial_attn) {
        add_wb(h, p + ".correlation.qkv.linear1", (int64_t)C * 9, C);
        add_wb(h, p + ".correlation.qkv.linear2", (int64_t)C * 9, C);
        add_wb(h, p + ".correlation.qkv.linear1_first", (int64_t)(C / 10) * C, C / 10);
        add_wb(h, p + ".correlation.qkv.linear1_second", (int64_t)C * (C / 10), C);
        add_wb(h, p + ".correlation.qkv.linear2_first", (int64_t)(C / 10) * C, C / 10);
        add_wb(h, p + ".correlation.qkv.linear2_second", (int64_t)C * (C / 10), C);
      }
      add_wb(h, p + ".correlation.proj", (int64_t)C * C, C);
      add_wb(h, p + ".correlation.spatial_linear", (int64_t)r * r, 1);
      add_wb(h, p + ".correlation.k_generate1", (int64_t)hd * hd, hd);
      add_wb(h, p + ".correlation.k_generate2", (int64_t)hd * hd, hd);
      add_wb(h, p + ".correlation.pos.pos_proj", (int64_t)pos_dim * 2, pos_dim);
      add_wb(h, p + ".correlation.pos.pos1.0", pos_dim, pos_dim);
      add_wb(h, p + ".correlation.pos.pos1.2", (int64_t)pos_dim * pos_dim, pos_dim);
      add_wb(h, p + ".correlation.pos.pos2.0", pos_dim, pos_dim);
      add_wb(h, p + ".correlation.pos.pos2.2", (int64_t)pos_dim * pos_dim, pos_dim);
      add_wb(h, p + ".correlation.pos.pos3.0", pos_dim, pos_dim);
      add_wb(h, p + ".correlation.pos.pos3.2", (int64_t)c.num_heads[i] * pos_dim, c.num_heads[i]);
      add_wb(h, p + ".norm2", C, C);
      add_wb(h, p + ".mlp.fc1", (int64_t)hidden * C, hidden);
      add_wb(h, p + ".mlp.dwconv.depthwise_conv.0", (int64_t)hidden * 25, hidden);
      add_wb(h, p + ".mlp.fc2", (int64_t)C * hidden, C);
    }
    if (c.resi_3conv) {
      const std::string p = "layers." + std::to_string(i) + ".conv";
      add_wb(h, p + ".0", (int64_t)(C / 4) * C * 9, C / 4);
      add_wb(h, p + ".2", (int64_t)(C / 4) * (C / 4), C / 4);
      add_wb(h, p + ".4", (int64_t)C * (C / 4) * 9, C);
    } else {
      add_wb(h, "layers." + std::to_string(i) + ".conv", (int64_t)C * C * 9, C);
    }
  }
  add_wb(h, "norm", C, C);
  if (c.resi_3conv) {
    add_wb(h, "conv_after_body.0", (int64_t)(C / 4) * C * 9, C / 4);
    add_wb(h, "conv_after_body.2", (int64_t)(C / 4) * (C / 4), C / 4);
    add_wb(h, "conv_after_body.4", (int64_t)C * (C / 4) * 9, C);
  } else {
    add_wb(h, "conv_after_body", (int64_t)C * C * 9, C);
  }
  const int s = c.upscale;
  switch (c.upsampler) {
    case HITSIR_UP_PIXELSHUFFLE:
      add_wb(h, "conv_before_upsample.0", (int64_t)kNumFeat * C * 9, kNumFeat);
      if ((s & (s - 1)) == 0) {
        int n = 0;
        for (int t = s; t > 1; t >>= 1) ++n;
        for (int k = 0; k < n; ++k) add_wb(h, "upsample." + std::to_string(2 * k), (int64_t)4 * kNumFeat * kNumFeat * 9, 4 * kNumFeat);
      } else {
        add_wb(h, "upsample.0", (int64_t)9 * kNumFeat * kNumFeat * 9, 9 * kNumFeat);
      }
      add_wb(h, "conv_last", (int64_t)ic * kNumFeat * 9, ic);
      break;
    case HITSIR_UP_PIXELSHUFFLEDIRECT:
      add_wb(h, "upsample.0", (int64_t)s * s * ic * C * 9, s * s * ic);
      break;
    case HITSIR_UP_NEAREST_CONV:
      add_wb(h, "conv_before_upsample.0", (int64_t)kNumFeat * C * 9, kNumFeat);
      add_wb(h, "conv_up1", (int64_t)kNumFeat * kNumFeat * 9, kNumFeat);
      add_wb(h, "conv_up2", (int64_t)kNumFeat * kNumFeat * 9, kNumFeat);
      add_wb(h, "conv_hr", (int64_t)kNumFeat * kNumFeat * 9, kNumFeat);
      add_wb(h, "conv_last", (int64_t)ic * kNumFeat * 9, ic);
      break;
    default:
      add_wb(h, "conv_last", (int64_t)ic * C * 9, ic);
      break;
  }
}

int validate_config(const HitsirConfig& c) {
  if (c.embed_dim != kC) { set_error("unsupported embed_dim %d: this build implements HiT-SIR-pro (embed_dim=180)", c.embed_dim); return HITSIR_ERR_UNSUPPORTED; }
  if (c.in_chans != 3 && c.in_chans != 1) { set_error("in_chans must be 1 or 3, got %d", c.in_chans); return HITSIR_ERR_UNSUPPORTED; }
  if (c.is_mult_size_conv_feat_extract && c.in_chans != 3) { set_error("MultipleSizeConvExtract needs in_chans == 3 (conv_x is Conv2d(3,..), hit_sir_pro.py:59)"); return HITSIR_ERR_UNSUPPORTED; }
  if (c.num_layers < 1 || c.num_layers > HITSIR_MAX_LAYERS) { set_error("num_layers %d out of range", c.num_layers); return HITSIR_ERR_INVALID; }
  if (c.mlp_ratio != 2.0f) { set_error("unsupported mlp_ratio %f (this build: 2.0)", c.mlp_ratio); return HITSIR_ERR_UNSUPPORTED; }
  if (c.base_win_size[0] != c.base_win_size[1] || c.base_win_size[0] < 1 || c.base_win_size[0] > 8) {
    set_error("unsupported base_win_size (%d,%d): square windows with base <= 8 only", c.base_win_size[0], c.base_win_size[1]);
    return HITSIR_ERR_UNSUPPORTED;
  }
  for (int i = 0; i < c.num_layers; ++i) {
    if (c.num_heads[i] != kHeads) { set_error("unsupported num_heads[%d]=%d (this build: 6)", i, c.num_heads[i]); return HITSIR_ERR_UNSUPPORTED; }
    if (c.depths[i] < 1 || c.depths[i] > c.num_ratios || c.depths[i] > HITSIR_MAX_DEPTH) {
      set_error("depths[%d]=%d needs that many hier_win_ratios (have %d)", i, c.depths[i], c.num_ratios);
      return HITSIR_ERR_INVALID;
    }
    for (int j = 0; j < c.depths[i]; ++j) {
      const int w = win_of(c, j), bs = c.base_win_size[0];
      if (w < 1) { set_error("window %d of block %d is empty", w, j); return HITSIR_ERR_INVALID; }
      // reference assertion, hit_sir_pro.py:647-649
      if (w > bs && w % bs != 0) { set_error("please ensure the window size is smaller than or divisible by the base window size"); return HITSIR_ERR_INVALID; }
      if (scc_tile(w).TT == 0) { set_error("window %d not supported by this build (4, 8, 16, 32, 48, 64)", w); return HITSIR_ERR_UNSUPPORTED; }
    }
  }
  if (c.upsampler == HITSIR_UP_NEAREST_CONV && c.upscale != 4) { set_error("only support x4 now."); return HITSIR_ERR_INVALID; }   // (:1248)
  if (c.upsampler == HITSIR_UP_PIXELSHUFFLE) {
    const int s = c.upscale;
    if (!((s & (s - 1)) == 0 || s == 3) || s < 1) { set_error("scale %d is not supported. Supported scales: 2^n and 3.", s); return HITSIR_ERR_INVALID; }   // (:1042)
    if (s > 4) { set_error("upsampler='pixelshuffle' with upscale %d is not implemented in this build (1, 2, 3, 4)", s); return HITSIR_ERR_UNSUPPORTED; }
  }
  if (c.upsampler == HITSIR_UP_PIXELSHUFFLEDIRECT && (c.upscale < 1 || c.upscale * c.upscale * c.in_chans > 256)) {
    set_error("pixelshuffledirect upscale %d not supported", c.upscale); return HITSIR_ERR_UNSUPPORTED;
  }
  if (c.ape_tokens < 0) { set_error("ape_tokens must be >= 0"); return HITSIR_ERR_INVALID; }
  return 0;
}

const float* P(const HitsirHandle* h, const std::string& name) {
  auto it = h->index.find(name);
  if (it == h->index.end()) return nullptr;
  return h->arena + h->params[it->second].offset;
}

constexpr size_t kPackChunkBytes = (size_t)64 << 20;
template <class T>
int dev_alloc(HitsirHandle* h, T** p, size_t count) {
  const size_t bytes = (count * sizeof(T) + 1023) & ~(size_t)1023;      // 1024: swizzled operand images are bulk-copied to 1024-byte aligned smem
  while (h->chunk_cur < h->owned.size() && h->chunk_off + bytes > h->chunk_bytes[h->chunk_cur]) { ++h->chunk_cur; h->chunk_off = 0; }
  if (h->chunk_cur == h->owned.size()) {
    const size_t cb = bytes > kPackChunkBytes ? bytes : kPackChunkBytes;
    void* q = nullptr;
    HITSIR_CHECK(cudaMalloc(&q, cb));
    h->owned.push_back(q);
    h->chunk_bytes.push_back(cb);
    h->chunk_off = 0;
  }
  *p = reinterpret_cast<T*>(static_cast<uint8_t*>(h->owned[h->chunk_cur]) + h->chunk_off);
  h->chunk_off += bytes;
  return 0;
}

int pick_bn(int n) {
  if (n <= 16) return 16;
  if (n <= 32) return 32;
  if (n <= 48) return 48;
  if (n <= 64) return 64;
  if (n % 256 == 0) return 256;
  return 192;
}

// conv (taps=9) or linear (taps=1) weight `prefix` -> packed GEMM operand
int make_gemm_w(HitsirHandle* h, GemmW* g, const std::string& prefix, int Co, int Ci, int taps, cudaStream_t st, int perm_k = 0) {
  const int BN = pick_bn(Co);
  const int Npad = round_up(Co, BN), Cipad = round_up(Ci, 64);
  g->BN = BN; g->Npad = Npad; g->K = taps * Cipad;
  if (dev_alloc(h, &g->w, (size_t)Npad * g->K)) return 1;
  if (dev_alloc(h, &g->b, (size_t)Npad)) return 1;
  const float* w = P(h, prefix + ".weight");
  const float* b = P(h, prefix + ".bias");
  if (!w || !b) { set_error("missing parameter %s", prefix.c_str()); return 1; }
  if (launch_pack_conv(w, b, g->w, g->b, Co, Ci, taps, Npad, Cipad, perm_k, st)) return 1;
  return make_tmap_2d(&g->tm, g->w, (uint64_t)g->K, (uint64_t)Npad, (uint64_t)g->K * 2, 64, (uint32_t)BN);
}

// conv_up1 / conv_up2 act on a x2 nearest-upsampled map: packed as the four 2x2 phase filters of the equivalent sub-pixel conv
int make_subpixel_w(HitsirHandle* h, GemmW* g, const std::string& prefix, cudaStream_t st) {
  g->BN = 64; g->Npad = 64; g->K = 16 * 64;
  if (dev_alloc(h, &g->w, (size_t)64 * g->K) || dev_alloc(h, &g->b, 64)) return 1;
  const float* w = P(h, prefix + ".weight");
  const float* b = P(h, prefix + ".bias");
  if (!w || !b) { set_error("missing parameter %s", prefix.c_str()); return 1; }
  if (launch_pack_subpixel(w, b, g->w, g->b, st)) return 1;
  return make_tmap_2d(&g->tm, g->w, (uint64_t)g->K, 64, (uint64_t)g->K * 2, 64, 64);
}

// conv_last over a 64-channel map: additionally the folded-tap operand of conv_last_fold_kernel
int make_last_w(HitsirHandle* h, GemmW* g, int ic, cudaStream_t st) {
  if (make_gemm_w(h, g, "conv_last", ic, kNumFeat, 9, st)) return 1;
  if (dev_alloc(h, &g->wf, (size_t)48 * 64)) return 1;
  if (launch_pack_fold_last(P(h, "conv_last.weight"), g->wf, ic, st)) return 1;
  return make_tmap_2d(&g->tmf, g->wf, 64, 48, 128, 64, 48);
}

void free_owned(HitsirHandle* h) {
  for (void* p : h->owned) cudaFree(p);
  h->owned.clear(); h->chunk_bytes.clear();
  h->chunk_cur = 0; h->chunk_off = 0;
}

int finalize(HitsirHandle* h, cudaStream_t st) {
  for (const ParamSpec& p : h->params)
    if (!p.set) { set_error("parameter '%s' was never provided (hitsir_set_param)", p.name.c_str()); return HITSIR_ERR_WEIGHTS; }
  // re-pack in place: the chunks are kept and refilled in the same order.  Work that still reads the old tables (possibly on another
  // stream) must have finished first -- cudaFree used to imply exactly this device-wide wait
  if (!h->owned.empty()) HITSIR_CHECK(cudaDeviceSynchronize());
  h->chunk_cur = 0; h->chunk_off = 0;
  h->finalized = false;
  const HitsirConfig& c = h->cfg;
  const int C = kC, ic = c.in_chans;
  // ---- shallow feature extraction
  if (c.is_mult_size_conv_feat_extract) {
    h->first_f = 9; h->first_kp = round_up(81 * ic, 64);
    GemmW& g = h->first;
    g.BN = 160; g.Npad = 960; g.K = h->first_kp;
    if (dev_alloc(h, &g.w, (size_t)960 * g.K) || dev_alloc(h, &g.b, 960)) return 1;
    if (launch_pack_msconv(P(h, "conv_first.conv3.weight"), P(h, "conv_first.conv5.weight"), P(h, "conv_first.conv7.weight"),
                           P(h, "conv_first.conv9.weight"), P(h, "conv_first.conv_x.weight"), P(h, "conv_first.conv3.bias"),
                           P(h, "conv_first.conv5.bias"), P(h, "conv_first.conv7.bias"), P(h, "conv_first.conv9.bias"),
                           P(h, "conv_first.conv_x.bias"), g.w, g.b, ic, g.K, st)) return 1;
    if (make_tmap_2d(&g.tm, g.w, (uint64_t)g.K, 960, (uint64_t)g.K * 2, 64, 160)) return 1;
    {
      GemmW& l = h->first_last;
      l.BN = 192; l.Npad = 192; l.K = 768;
      if (dev_alloc(h, &l.w, (size_t)192 * 768) || dev_alloc(h, &l.b, 192)) return 1;
      if (launch_pack_mslast(P(h, "conv_first.conv_last.weight"), P(h, "conv_first.conv_last.bias"), l.w, l.b, 192, st)) return 1;
      if (make_tmap_2d(&l.tm, l.w, 768, 192, 768 * 2, 64, 192)) return 1;
    }
  } else {
    h->first_f = 3; h->first_kp = round_up(9 * ic, 64);
    GemmW& g = h->first;
    g.BN = 192; g.Npad = 192; g.K = h->first_kp;
    if (dev_alloc(h, &g.w, (size_t)192 * g.K) || dev_alloc(h, &g.b, 192)) return 1;
    if (launch_pack_firstconv(P(h, "conv_first.weight"), P(h, "conv_first.bias"), g.w, g.b, C, ic, 3, g.K, st)) return 1;
    if (make_tmap_2d(&g.tm, g.w, (uint64_t)g.K, 192, (uint64_t)g.K * 2, 64, 192)) return 1;
  }
  // ---- blocks
  h->blocks.assign(c.num_layers, std::vector<BlockW>());
  h->layer_conv.assign(c.num_layers, GemmW());
  float* tbl_scratch = nullptr;
  if (dev_alloc(h, &tbl_scratch, (size_t)127 * 127 * kHeads)) return 1;
  for (int i = 0; i < c.num_layers; ++i) {
    h->blocks[i].resize(c.depths[i]);
    for (int j = 0; j < c.depths[i]; ++j) {
      BlockW& bw = h->blocks[i][j];
      const std::string p = "layers." + std::to_string(i) + ".residual_group.blocks." + std::to_string(j);
      bw.win = win_of(c, j);
      bw.base = bw.win < c.base_win_size[0] ? bw.win : c.base_win_size[0];
      bw.r = bw.win / bw.base;
      bw.g1 = P(h, p + ".norm1.weight"); bw.b1 = P(h, p + ".norm1.bias");
      bw.g2 = P(h, p + ".norm2.weight"); bw.b2 = P(h, p + ".norm2.bias");
      if (c.is_channel_spatial_attn) {
        const std::string q = p + ".correlation.qkv";
        if (dev_alloc(h, &bw.casa_w1, 9 * C) || dev_alloc(h, &bw.casa_w2, 9 * C)) return 1;
        if (launch_pack_tapmajor(P(h, q + ".linear1.weight"), bw.casa_w1, C, 9, C, st)) return 1;
        if (launch_pack_tapmajor(P(h, q + ".linear2.weight"), bw.casa_w2, C, 9, C, st)) return 1;
        bw.casa.w1 = bw.casa_w1; bw.casa.b1 = P(h, q + ".linear1.bias");
        bw.casa.w2 = bw.casa_w2; bw.casa.b2 = P(h, q + ".linear2.bias");
        bw.casa.l1f_w = P(h, q + ".linear1_first.weight"); bw.casa.l1f_b = P(h, q + ".linear1_first.bias");
        bw.casa.l1s_w = P(h, q + ".linear1_second.weight"); bw.casa.l1s_b = P(h, q + ".linear1_second.bias");
        bw.casa.l2f_w = P(h, q + ".linear2_first.weight"); bw.casa.l2f_b = P(h, q + ".linear2_first.bias");
        bw.casa.l2s_w = P(h, q + ".linear2_second.weight"); bw.casa.l2s_b = P(h, q + ".linear2_second.bias");
        bw.casa.bfrag = nullptr;
        if (dev_alloc(h, &bw.casa_bfrag, (size_t)casa_bfrag_words())) return 1;
        if (launch_pack_casa_bfrag(bw.casa, bw.casa_bfrag, st)) return 1;
        bw.casa.bfrag = bw.casa_bfrag;
      }
      const std::string s = p + ".correlation";
      bw.scc.wk1 = P(h, s + ".k_generate1.weight"); bw.scc.bk1 = P(h, s + ".k_generate1.bias");
      bw.scc.wk2 = P(h, s + ".k_generate2.weight"); bw.scc.bk2 = P(h, s + ".k_generate2.bias");
      bw.scc.wsl = P(h, s + ".spatial_linear.weight");
      bw.scc.bsl_dev = const_cast<float*>(P(h, s + ".spatial_linear.bias"));
      PosW pw;
      pw.proj_w = P(h, s + ".pos.pos_proj.weight"); pw.proj_b = P(h, s + ".pos.pos_proj.bias");
      for (int k = 0; k < 3; ++k) {
        const std::string pk = s + ".pos.pos" + std::to_string(k + 1);
        pw.ln_w[k] = P(h, pk + ".0.weight"); pw.ln_b[k] = P(h, pk + ".0.bias");
        pw.fc_w[k] = P(h, pk + ".2.weight"); pw.fc_b[k] = P(h, pk + ".2.bias");
      }
      const int L = bw.win * bw.win, Lb = bw.base * bw.base;
      if (dev_alloc(h, &bw.bias_tbl, (size_t)kHeads * L * Lb)) return 1;
      if (launch_pos_table(pw, bw.win, tbl_scratch, st)) return 1;
      if (launch_pooled_bias(tbl_scratch, bw.win, bw.base, bw.bias_tbl, st)) return 1;
      bw.scc.bias_tbl = bw.bias_tbl;
      if (dev_alloc(h, &bw.pool_img, scc_pool_image_bytes(bw.win)) || dev_alloc(h, &bw.bias_img, scc_bias_image_bytes(bw.win)) ||
          dev_alloc(h, &bw.w_img, 2048)) return 1;
      if (launch_scc_images(bw.scc, bw.win, bw.base, bw.pool_img, bw.bias_img, bw.w_img, st)) return 1;
      bw.scc.pool_img = bw.pool_img; bw.scc.bias_img = bw.bias_img; bw.scc.w_img = bw.w_img;
      // proj consumes the SCC output in its head-padded channel order (kernels.cuh scc_pos)
      if (make_gemm_w(h, &bw.proj, s + ".proj", C, C, 1, st, 1)) return 1;
      if (make_gemm_w(h, &bw.fc1, p + ".mlp.fc1", kHid, C, 1, st)) return 1;
      if (make_gemm_w(h, &bw.fc2, p + ".mlp.fc2", C, kHid, 1, st)) return 1;
      // [26][384] fp32: 25 tap rows + the bias as row 25 (one TMA box per 64-channel slice in ffn_tail.cu)
      if (dev_alloc(h, &bw.dw_w, 26 * kHidp)) return 1;
      bw.dw_b = bw.dw_w + 25 * kHidp;
      if (launch_pack_tapmajor(P(h, p + ".mlp.dwconv.depthwise_conv.0.weight"), bw.dw_w, kHid, 25, kHidp, st)) return 1;
      if (launch_pack_tapmajor(P(h, p + ".mlp.dwconv.depthwise_conv.0.bias"), bw.dw_b, kHid, 1, kHidp, st)) return 1;
      if (dev_alloc(h, &bw.dw_mma, 28 * kHidp)) return 1;
      if (launch_pack_dw_mma(bw.dw_w, bw.dw_mma, st)) return 1;
      if (bw.fc2.Npad != 192 || bw.fc2.K != kHidp) { set_error("fc2 packing %d x %d is not the 192 x 384 the FFN tail expects", bw.fc2.Npad, bw.fc2.K); return 1; }
      if (dev_alloc(h, &bw.w2_img, (size_t)6 * 192 * 128)) return 1;
      if (launch_pack_w2_image(bw.fc2.w, bw.w2_img, st)) return 1;
    }
    if (!c.resi_3conv && make_gemm_w(h, &h->layer_conv[i], "layers." + std::to_string(i) + ".conv", C, C, 9, st)) return 1;
  }
  if (c.resi_3conv) {
    h->r3_a.assign(c.num_layers + 1, GemmW()); h->r3_b.assign(c.num_layers + 1, GemmW()); h->r3_c.assign(c.num_layers + 1, GemmW());
    for (int i = 0; i <= c.num_layers; ++i) {
      const std::string p = i < c.num_layers ? "layers." + std::to_string(i) + ".conv" : std::string("conv_after_body");
      if (make_gemm_w(h, &h->r3_a[i], p + ".0", C / 4, C, 9, st)) return 1;
      if (make_gemm_w(h, &h->r3_b[i], p + ".2", C / 4, C / 4, 1, st)) return 1;
      if (make_gemm_w(h, &h->r3_c[i], p + ".4", C, C / 4, 9, st)) return 1;
    }
  } else if (make_gemm_w(h, &h->conv_after_body, "conv_after_body", C, C, 9, st)) return 1;
  if (c.is_fusion) {
    for (int u = 0; u < 3; ++u) {
      const std::string p = "fusion.union_attention" + std::to_string(u + 1);
      h->ua[u].small.c1_w = P(h, p + ".conv1.weight"); h->ua[u].small.c1_b = P(h, p + ".conv1.bias");
      h->ua[u].small.c2_w = P(h, p + ".conv2.weight"); h->ua[u].small.c2_b = P(h, p + ".conv2.bias");
      h->ua[u].small.c3_w = P(h, p + ".conv3.weight"); h->ua[u].small.c3_b = P(h, p + ".conv3.bias");
      if (make_gemm_w(h, &h->ua[u].conv_last, p + ".conv_last", C, C, 9, st)) return 1;
    }
  }
  h->upsample.clear();
  const int s = c.upscale;
  switch (c.upsampler) {
    case HITSIR_UP_PIXELSHUFFLE: {
      if (make_gemm_w(h, &h->conv_before_upsample, "conv_before_upsample.0", kNumFeat, C, 9, st)) return 1;
      if ((s & (s - 1)) == 0) {
        int n = 0;
        for (int t = s; t > 1; t >>= 1) ++n;
        h->upsample.resize(n);
        for (int k = 0; k < n; ++k)
          if (make_gemm_w(h, &h->upsample[k], "upsample." + std::to_string(2 * k), 4 * kNumFeat, kNumFeat, 9, st)) return 1;
      } else {
        h->upsample.resize(1);
        if (make_gemm_w(h, &h->upsample[0], "upsample.0", 9 * kNumFeat, kNumFeat, 9, st)) return 1;
      }
      if (make_last_w(h, &h->conv_last, ic, st)) return 1;
      break;
    }
    case HITSIR_UP_PIXELSHUFFLEDIRECT:
      h->upsample.resize(1);
      if (make_gemm_w(h, &h->upsample[0], "upsample.0", s * s * ic, C, 9, st)) return 1;
      break;
    case HITSIR_UP_NEAREST_CONV:
      if (make_gemm_w(h, &h->conv_before_upsample, "conv_before_upsample.0", kNumFeat, C, 9, st)) return 1;
      if (make_subpixel_w(h, &h->conv_up1, "conv_up1", st)) return 1;
      if (make_subpixel_w(h, &h->conv_up2, "conv_up2", st)) return 1;
      if (make_gemm_w(h, &h->conv_hr, "conv_hr", kNumFeat, kNumFeat, 9, st)) return 1;
      if (make_last_w(h, &h->conv_last, ic, st)) return 1;
      break;
    default:
      if (make_gemm_w(h, &h->conv_last, "conv_last", ic, C, 9, st)) return 1;
      break;
  }
  h->finalized = true;
  return 0;
}

// ------------------------------------------------------------------------------------------
// workspace layout
// ------------------------------------------------------------------------------------------
struct Workspace {
  size_t bytes = 0;
  float *P = nullptr, *Q = nullptr, *S = nullptr;        // fp32 [N,180]: layer stream, working stream, shallow features
  bf16 *xb0 = nullptr, *xb1 = nullptr;                   // bf16 [N,192] shadows (contiguous: also A0 [N,<=384])
  bf16* T = nullptr;                                     // bf16 [NpMax,192] qkv tokens on the padded map
  float *cavg = nullptr, *cmax = nullptr;                // [NpMax]
  float *part_sum = nullptr, *part_max = nullptr, *s1 = nullptr, *s2 = nullptr;
  float* scc_dbg = nullptr;
  bf16* outsc = nullptr;                                 // bf16 [N,192]
  bf16 *H1 = nullptr, *H2 = nullptr;                     // bf16 [N,384] (contiguous: also G [N,768], A1|A2 fp32)
  float *havg, *hmax, *wavg, *wmax, *c_att, *h_att, *w_att;
  float* red = nullptr;
  bf16* up = nullptr;                                    // upsampler scratch
  size_t up_bytes = 0;
  int nparts = 1;
};

struct Bump {
  uint8_t* base; size_t off = 0;
  template <class T> T* take(size_t count) {
    off = (off + 255) & ~(size_t)255;
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += count * sizeof(T);
    return p;
  }
  // `count` elements with `halo` extra elements reserved in front of and behind them (band mode: rows exchanged with the neighbour
  // bands); returns the first CORE element.  The halo is rounded up so that the core stays 256-byte aligned.
  template <class T> T* take_ext(size_t count, size_t halo) {
    const size_t hb = (halo * sizeof(T) + 255) & ~(size_t)255;
    off = (off + 255) & ~(size_t)255;
    T* p = base ? reinterpret_cast<T*>(base + off + hb) : nullptr;
    off += 2 * hb + count * sizeof(T);
    return p;
  }
};

// `halo`: 0 = ordinary forward; > 0 = band mode (exact row sharding of one frame): every buffer that a vertical stencil reads gets room
// for halo rows above and below (at most 2 rows of its own row size), and H is the LARGEST band height of the frame so that every
// rank / band lays its workspace out identically (peer addresses = own base + same offset)
int layout_workspace(const HitsirHandle* h, int B, int H, int W, void* base, Workspace* ws, int halo = 0) {
  const HitsirConfig& c = h->cfg;
  const size_t N = (size_t)B * H * W;
  size_t np_max = N;
  int max_depth = 0;
  for (int i = 0; i < c.num_layers; ++i) max_depth = c.depths[i] > max_depth ? c.depths[i] : max_depth;
  for (int j = 0; j < max_depth; ++j) {
    const int w = win_of(c, j);
    const int Hp = round_up(H, w), Wp = round_up(W, w);
    if (Hp - H >= H || Wp - W >= W) {
      set_error("Padding size should be less than the corresponding input dimension, but got: padding (%d, %d) for input %dx%d (window %d)",
                Wp - W, Hp - H, H, W, w);
      return HITSIR_ERR_INPUT_TOO_SMALL;
    }
    const size_t np = (size_t)B * Hp * Wp;
    np_max = np > np_max ? np : np_max;
  }
  Bump b{reinterpret_cast<uint8_t*>(base)};
  ws->P = b.take<float>(N * kC);
  ws->Q = b.take<float>(N * kC);
  ws->S = b.take<float>(N * kC);
  const size_t hr = halo ? (size_t)W : 0;     // one halo row = W pixels
  if (!halo) {
    ws->xb0 = b.take<bf16>(N * kCp * 2);   // xb0 | xb1 contiguous
    ws->xb1 = ws->xb0 ? ws->xb0 + N * kCp : nullptr;
  } else {
    ws->xb0 = b.take_ext<bf16>(N * kCp * 2, hr * kCp);       // also holds the im2col rows [N, <= 384]
    ws->xb1 = b.take_ext<bf16>(N * kCp, hr * kCp);
  }
  ws->T = b.take<bf16>(np_max * kCp);
  ws->cavg = b.take_ext<float>(np_max, hr);
  ws->cmax = b.take_ext<float>(np_max, hr);
  ws->nparts = 64;
  {
    const size_t np = (size_t)(ffn_tiles_per_image(H, W) > ws->nparts ? ffn_tiles_per_image(H, W) : ws->nparts);   // ffn_tail emits one partial per 8x16 tile
    ws->part_sum = b.take<float>((size_t)B * np * kC);
    ws->part_max = b.take<float>((size_t)B * np * kC);
  }
  ws->s1 = b.take<float>((size_t)B * kC);
  ws->s2 = b.take<float>((size_t)B * kC);
  ws->scc_dbg = b.take<float>((size_t)kSccDbgFloats);
  ws->outsc = b.take_ext<bf16>(N * kCp, hr * kCp);
  ws->H1 = b.take_ext<bf16>(N * kHidp * 2, 2 * hr * kHidp);  // H1 | H2 contiguous
  ws->H2 = ws->H1 ? ws->H1 + N * kHidp : nullptr;
  ws->havg = b.take<float>((size_t)B * kC * W * 2);           // havg | hmax contiguous (one all-reduce payload each, adjacent)
  ws->hmax = ws->havg ? ws->havg + (size_t)B * kC * W : nullptr;
  ws->wavg = b.take_ext<float>((size_t)B * kC * H, halo ? kC : 0);
  ws->wmax = b.take_ext<float>((size_t)B * kC * H, halo ? kC : 0);
  ws->red = b.take<float>(2 * kCp);                           // band mode: [sum 180 | pad][max 180 | pad] all-reduce payload of the casa pools
  ws->c_att = b.take<float>(N);
  ws->h_att = b.take<float>((size_t)B * kC * W);
  ws->w_att = b.take<float>((size_t)B * kC * H);
  // upsampler scratch (bf16 elements)
  size_t up = 0;
  const int s = c.upscale;
  switch (c.upsampler) {
    case HITSIR_UP_NEAREST_CONV: up = N * kNumFeat * (size_t)(1 + 4 + 16 + 16); break;   // U0, U1, U2, U3 (no replicated maps: launch_conv3_c64_up)
    case HITSIR_UP_PIXELSHUFFLE: up = N * kNumFeat * (size_t)(1 + 4 + (s > 2 ? s * s : 0)); break;
    default: up = 0; break;
  }
  if (halo) up += (size_t)16 * 2 * 4 * W * kNumFeat;          // halo rows of the (at most five) upsampler maps, each <= 2 rows of 4W pixels
  ws->up_bytes = up * sizeof(bf16);
  ws->up = b.take<bf16>(up);
  ws->bytes = (b.off + 255) & ~(size_t)255;
  return 0;
}

// ------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------
struct Fwd {
  HitsirHandle* h;
  cudaStream_t st;
  int B, H, W;
  long long N;
  Workspace ws;
  bool stopped = false;
  int stats_nparts = 0;      // > 0: casa statistics of the current stream were produced by the previous block's ffn_tail (partials per image)
  // band mode (hitsir_forward_band): this call computes rows [row0, row0 + H) of a frame with Hf rows; halos come from the callbacks
  const HitsirBand* band = nullptr;
  void* ws_base = nullptr;
  long long Nl = 0;          // pixels of the workspace LAYOUT (= N; band mode: B * layout_h * W, so that sub-buffers sit at the same offsets in every band)
  int row0 = 0, Hf = 0;
  bool top = false, bot = false;     // a neighbour band exists above / below
};

// Make the `halo` rows above and below the `rows` core rows of a row-major buffer valid before a vertical stencil reads them: rows
// outside the frame are zero (the stencil's zero padding), rows of a neighbour band are fetched through the caller's exchange callback
// (which runs on the host while the forward is being enqueued and must order its copies on `stream`).  No-op outside band mode.
int fill_halo(Fwd& f, void* core, size_t row_bytes, int rows, int halo) {
  if (f.band == nullptr) return 0;
  uint8_t* c = reinterpret_cast<uint8_t*>(core);
  if (!f.top) HITSIR_CHECK(cudaMemsetAsync(c - (size_t)halo * row_bytes, 0, (size_t)halo * row_bytes, f.st));
  if (!f.bot) HITSIR_CHECK(cudaMemsetAsync(c + (size_t)rows * row_bytes, 0, (size_t)halo * row_bytes, f.st));
  if (f.top || f.bot) {
    const int rc = f.band->halo(f.band->ctx, (int64_t)(c - reinterpret_cast<uint8_t*>(f.ws_base)), (int64_t)row_bytes, rows, halo, f.st);
    if (rc) { set_error("band halo exchange callback failed (%d)", rc); return HITSIR_ERR_INVALID; }
  }
  return 0;
}
// element-wise SUM of `n_sum` floats at `sum` and MAX of `n_max` floats at `mx` over all bands of the frame (in place)
int band_allreduce(Fwd& f, float* sum, int64_t n_sum, float* mx, int64_t n_max) {
  if (f.band == nullptr || f.band->allreduce == nullptr) return 0;     // a single band still reports its statistics when a callback is given
  uint8_t* b0 = reinterpret_cast<uint8_t*>(f.ws_base);
  const int rc = f.band->allreduce(f.band->ctx, (int64_t)(reinterpret_cast<uint8_t*>(sum) - b0), n_sum, (int64_t)(reinterpret_cast<uint8_t*>(mx) - b0), n_max, f.st);
  if (rc) { set_error("band all-reduce callback failed (%d)", rc); return HITSIR_ERR_INVALID; }
  return 0;
}

// returns 1 on error, sets f.stopped when the requested tap asked to stop
int do_tap(Fwd& f, const char* name, const void* src, int is_bf16, int ld, long long rows, int cols, int perm = 0) {
  Tap& t = f.h->tap;
  if (t.dst == nullptr || t.name != name) return 0;
  if (rows * cols > t.floats) { set_error("tap '%s' needs %lld floats, destination has %lld", name, rows * cols, (long long)t.floats); return HITSIR_ERR_INVALID; }
  if (launch_f32_to_f32_tap(src, is_bf16, ld, t.dst, rows, cols, perm, f.st)) return 1;
  if (t.stop) f.stopped = true;
  return 0;
}

// `name` matches the pending injection: overwrite the fp32 rows [rows, 180] at `dst_f32` and/or the bf16 rows [rows, 192] at `dst_bf16`
int do_inject(Fwd& f, const char* name, float* dst_f32, bf16* dst_bf16, long long rows) {
  Inject& in = f.h->inject;
  if (in.src == nullptr || in.name != name) return 0;
  if (rows * kC != in.floats) { set_error("inject '%s' needs %lld floats, source has %lld", name, rows * kC, (long long)in.floats); return HITSIR_ERR_INVALID; }
  if (dst_f32 != nullptr) HITSIR_CHECK(cudaMemcpyAsync(dst_f32, in.src, (size_t)rows * kC * sizeof(float), cudaMemcpyDeviceToDevice, f.st));
  if (dst_bf16 != nullptr && launch_cast_rows_bf16(in.src, dst_bf16, rows, f.st)) return 1;
  return 0;
}

#define RUN(expr) do { int _r = (expr); if (_r) return _r; } while (0)
struct ProfScope {
  HitsirHandle* h; cudaStream_t st; int idx = -1;
  ProfScope(HitsirHandle* h_, cudaStream_t st_, const char* cat) : h(h_), st(st_) {
    if (!h->prof.on) return;
    ProfRec r{h->prof.cat_id(cat), h->prof.get(), h->prof.get()};
    cudaEventRecord(r.a, st);
    h->prof.recs.push_back(r);
    idx = (int)h->prof.recs.size() - 1;
  }
  ~ProfScope() { if (idx >= 0) cudaEventRecord(h->prof.recs[idx].b, st); }
};
// one (or n) kernel launch(es) of category `cat`
#define LAUNCH(cat, n, expr) do { ProfScope _ps(f.h, f.st, cat); f.h->launches += (n); int _r = (expr); if (_r) return _r; } while (0)
void base_params(GemmParams& p, const GemmW& w) {
  memset(&p, 0, sizeof(p));
  p.n_tiles = w.Npad / w.BN;
  p.num_kb = w.K / 64;
  p.cblocks = p.num_kb;
  p.bias = w.b;
  p.Wp = w.w; p.ldw = w.K;
  p.ps = 1;
  p.slope = 1.f;
}

// The staged-epilogue kernel covers the plain-store and LayerNorm epilogues; the gate / pixel-shuffle
// epilogues (once per forward) keep the direct-store kernel.
bool tma_epilogue(const HitsirHandle* h, const GemmW& w, const GemmParams& p) {
  if (h->simt || h->direct_epilogue) return false;
  if (p.epi == EPI_MSGATE) return w.BN == 160;
  return (p.epi == EPI_STORE || p.epi == EPI_LN) && (w.BN == 192 || w.BN == 64) && p.out2_f32 == nullptr && w.Npad <= 384;
}

int run_gemm(Fwd& f, const char* cat, const GemmW& w, GemmParams& p, const CUtensorMap* maps, bool tma) {
  ProfScope ps(f.h, f.st, cat);
  f.h->launches++;
#ifdef HITSIR_AB_PATHS
  if (f.h->simt) return launch_simt_gemm(w.BN, p, f.st);
#endif
  if (tma) return launch_umma_gemm_tma(w.BN, p, maps, f.h->num_sms, f.st);
  return launch_umma_gemm(w.BN, p, maps[0], w.tm, f.h->num_sms, f.st);
}

// token-major linear: A [M, lda] bf16 (lda == w.K)
int linear(Fwd& f, const char* cat, const GemmW& w, const bf16* A, long long M, GemmParams& p) {
  p.conv = 0; p.M = (int)M; p.m_tiles = (int)cdiv64(M, 128);
  p.A = A; p.lda = w.K;
  p.b_resident = f.h->b_streamed ? 0 : 1;                  // honoured by the TMA kernel when the weight tile fits next to the A ring

  CUtensorMap maps[5];
  const bool tma = tma_epilogue(f.h, w, p);
  if (!f.h->simt) {
    if (make_tmap_2d(&maps[0], A, (uint64_t)w.K, (uint64_t)M, (uint64_t)w.K * 2, 64, 128)) return 1;
    maps[1] = w.tm; maps[2] = maps[0]; maps[3] = maps[0]; maps[4] = maps[0];
    if (tma) {
      if (p.out_f32 && make_tmap_2d_t(&maps[2], p.out_f32, 4, (uint64_t)p.n_real, (uint64_t)M, (uint64_t)p.ldf * 4, 32, 128)) return 1;
      if (p.out_bf16 && make_tmap_2d_t(&maps[3], p.out_bf16, 2, (uint64_t)p.ldb, (uint64_t)M, (uint64_t)p.ldb * 2, 64, 128)) return 1;
      if (p.res && make_tmap_2d_t(&maps[4], p.res, 4, (uint64_t)p.n_real, (uint64_t)M, (uint64_t)p.ldr * 4, 32, 128)) return 1;
    }
  }
  return run_gemm(f, cat, w, p, maps, tma);
}

// 3x3 conv over NHWC bf16 [B,H,W,Cpad].  Band mode: the rows above / below A are made valid first (fill_halo: zeros at the frame
// border, the neighbour band's rows otherwise) and the A tensor map starts one row above image row 0.
int conv3(Fwd& f, const char* cat, const GemmW& w, const bf16* A, int B, int H, int W, int Cpad, GemmParams& p) {
  p.conv = 1; p.B = B; p.H = H; p.W = W;
  if (f.band != nullptr) {
    RUN(fill_halo(f, const_cast<bf16*>(A), (size_t)W * Cpad * sizeof(bf16), H, 1));
    p.a_y_off = 1;
  }
  p.tiles_x = cdiv(W, 16); p.tiles_y = cdiv(H, 8);
  p.m_tiles = B * p.tiles_x * p.tiles_y;
  p.cblocks = Cpad / 64;
  p.A = A; p.lda = Cpad;
  if (w.K != 9 * Cpad) { set_error("conv3: packed K %d != 9*%d", w.K, Cpad); return 1; }
  // 64-channel inputs (HR stage): resident filter bank + kx-shared halo boxes (conv3_c64.cu)
  if (!f.h->simt && !f.h->direct_epilogue && Cpad == 64 && p.res == nullptr && p.out2_f32 == nullptr &&
      ((w.BN == 64 && p.epi == EPI_STORE && p.out_bf16 != nullptr && p.out_f32 == nullptr && p.ldb == 64) ||
       (w.BN == 16 && w.wf != nullptr && p.res_img == nullptr && p.epi == EPI_SHUFFLE_NCHW && p.ps == 1 && p.n_real <= 4))) {
    ProfScope ps(f.h, f.st, cat);
    f.h->launches++;
    if (w.BN == 16) return launch_conv_last_fold(p, A, w.tmf, f.h->num_sms, f.st);
    return launch_conv3_c64(w.BN, p, A, w.tm, f.h->num_sms, f.st);
  }
  CUtensorMap maps[5];
  const bool tma = tma_epilogue(f.h, w, p);
  if (!f.h->simt) {
    if (make_tmap_nhwc(&maps[0], A - (size_t)p.a_y_off * W * Cpad, B, H + 2 * p.a_y_off, W, Cpad, 64, 16, 8)) return 1;
    maps[1] = w.tm; maps[2] = maps[0]; maps[3] = maps[0]; maps[4] = maps[0];
    if (tma) {
      if (p.out_f32 && make_tmap_nhwc_t(&maps[2], p.out_f32, 4, B, H, W, p.n_real, p.ldf, 32, 16, 8)) return 1;
      if (p.out_bf16 && make_tmap_nhwc_t(&maps[3], p.out_bf16, 2, B, H, W, p.ldb, p.ldb, 64, 16, 8)) return 1;
      if (p.res && make_tmap_nhwc_t(&maps[4], p.res, 4, B, H, W, p.n_real, p.ldr, 32, 16, 8)) return 1;
    }
  }
  return run_gemm(f, cat, w, p, maps, tma);
}

// x2 nearest upsampling + 3x3 conv 64 -> 64 (+ LeakyReLU) on the LR map A [B,H,W,64] -> out [B,2H,2W,64] (:1331-1332).  Band mode: the
// LR rows above / below the band are exchanged (one LR row is what the replicated map's halo row was made of)
int conv3_up(Fwd& f, const char* cat, const GemmW& w, const bf16* A, int B, int H, int W, GemmParams& p) {
  p.conv = 1; p.B = B; p.H = H; p.W = W;
  if (f.band != nullptr) {
    RUN(fill_halo(f, const_cast<bf16*>(A), (size_t)W * kNumFeat * sizeof(bf16), H, 1));
    p.a_y_off = 1;
  }
  p.tiles_x = cdiv(W, 16); p.tiles_y = cdiv(H, 8);
  p.m_tiles = B * p.tiles_x * p.tiles_y;
  p.cblocks = 1;
  p.A = A; p.lda = kNumFeat;
  if (w.K != 16 * kNumFeat) { set_error("conv3_up: packed K %d is not the sub-pixel layout", w.K); return 1; }
  ProfScope ps(f.h, f.st, cat);
  f.h->launches++;
  return launch_conv3_c64_up(p, A, w.tm, f.h->num_sms, f.st);
}

#define TAP(name, src, is_bf16, ld, rows, cols) do { RUN(do_tap(f, name, src, is_bf16, ld, rows, cols)); if (f.stopped) return 0; } while (0)
#define TAPP(name, src, is_bf16, ld, rows, cols) do { RUN(do_tap(f, name, src, is_bf16, ld, rows, cols, 1)); if (f.stopped) return 0; } while (0)

int forward_block(Fwd& f, int i, int j, float* xin, float* xout) {
  // HierarchicalTransformerBlock.forward (:676-706); xin -> xout after the attention half, then in place on xout
  HitsirHandle* h = f.h;
  const HitsirConfig& c = h->cfg;
  Workspace& ws = f.ws;
  const BlockW& bw = h->blocks[i][j];
  const std::string tn = "block" + std::to_string(i) + "." + std::to_string(j);
  const int w = bw.win;
  SccGeom g;
  g.pg = PadGeom{f.B, f.H, f.W, round_up(f.H, w), round_up(f.W, w)};
  if (f.band != nullptr) {     // frame-level geometry of the casa pools and the neighbours' statistic rows (kernels.cuh PadGeom)
    g.pg.y0 = f.row0; g.pg.Hf = f.Hf; g.pg.Hpf = round_up(f.Hf, w);
    g.pg.top = f.top ? 1 : 0; g.pg.bot = (f.bot && g.pg.Hp == f.H) ? 1 : 0;
  }
  g.w = w; g.base = bw.base; g.r = bw.r; g.L = w * w; g.Lb = bw.base * bw.base;
  g.nWy = g.pg.Hp / w; g.nWx = g.pg.Wp / w; g.parts = 1;
  const long long Np = (long long)f.B * g.pg.Hp * g.pg.Wp;
  {
    const Inject& in = h->inject;
    if (in.src != nullptr && in.name == tn + ".in") {
      RUN(do_inject(f, in.name.c_str(), xin, nullptr, f.N));
      f.stats_nparts = 0;                                  // statistics delivered by the previous block no longer describe the stream
    }
  }
  if (c.is_channel_spatial_attn) {
    int nparts = f.stats_nparts;
    if (nparts == 0) {       // no producer epilogue delivered them (first block of a layer, unfused fallback): one pass over the stream
      nparts = ws.nparts;
      LAUNCH("sca_stats", 1, launch_sca_stats(xin, g.pg, ws.cavg, ws.cmax, ws.part_sum, ws.part_max, nparts, f.st));
    }
    if (f.band != nullptr) {
      // the global pools run over the whole padded FRAME: reduce this band's partials to one (sum, max) pair per channel, all-reduce
      LAUNCH("sca_reduce", 1, launch_reduce_parts(ws.part_sum, ws.part_max, nparts, ws.red, ws.red + kCp, f.st));
      RUN(band_allreduce(f, ws.red, kC, ws.red + kCp, kC));
      LAUNCH("sca_mlp", 1, launch_sca_mlp(ws.red, ws.red + kCp, 1, g.pg, bw.casa, ws.s1, ws.s2, f.st));
      RUN(fill_halo(f, ws.cavg, (size_t)f.W * sizeof(float), f.H, 1));      // the 3x3 gate convs read the neighbours' statistic rows
      RUN(fill_halo(f, ws.cmax, (size_t)f.W * sizeof(float), f.H, 1));
    } else {
      LAUNCH("sca_mlp", 1, launch_sca_mlp(ws.part_sum, ws.part_max, nparts, g.pg, bw.casa, ws.s1, ws.s2, f.st));
    }
  }
  f.stats_nparts = 0;
  LAUNCH("qkv_build", 1, launch_qkv_build(xin, g.pg, c.is_channel_spatial_attn, ws.cavg, ws.cmax, ws.s1, ws.s2, bw.casa, ws.T, f.st));
  TAPP((tn + ".qkv").c_str(), ws.T, 1, kCp, Np, kC);
  {
    const bool want_dbg = h->tap.dst != nullptr && h->tap.name == tn + ".sccdbg";
    char cat[16]; snprintf(cat, sizeof(cat), "scc_w%d", w);
    if (g.r == 1 && !want_dbg && !h->scc_gram_only)
      LAUNCH(cat, 1, launch_scc_dense(ws.T, g, bw.scc, ws.outsc, h->num_sms, f.st));
    else
      LAUNCH(cat, 1, launch_scc_umma(ws.T, g, bw.scc, ws.outsc, want_dbg ? ws.scc_dbg : nullptr, h->num_sms, f.st));
  }
  TAP((tn + ".sccdbg").c_str(), ws.scc_dbg, 0, kSccDbgFloats, 1, kSccDbgFloats);
  TAPP((tn + ".scc").c_str(), ws.outsc, 1, kCp, f.N, kC);
  GemmParams p;
#ifdef HITSIR_AB_PATHS
  if (!h->simt && !h->direct_epilogue && h->projfc1_fused && bw.proj.BN == 192 && bw.proj.K == 192 && bw.fc1.K == 192 && bw.fc1.Npad == 384) {
    // proj + norm1 + residual and fc1 + GELU in one kernel (:597, :700-703, :39-41)
    LAUNCH("proj_fc1", 1, launch_proj_fc1(ws.outsc, bw.proj.tm, bw.proj.b, bw.g1, bw.b1, xin, xout, bw.fc1.w, bw.fc1.b, ws.H1, f.N, h->num_sms, f.st));
    TAP((tn + ".attn").c_str(), xout, 0, kC, f.N, kC);
  } else
#endif
  {
  // proj + norm1 + residual (:597, :700-703)
  base_params(p, bw.proj);
  p.epi = EPI_LN; p.n_real = kC; p.gamma = bw.g1; p.beta = bw.b1; p.res = xin; p.ldr = kC;
  p.out_f32 = xout; p.ldf = kC; p.out_bf16 = ws.xb0; p.ldb = kCp;
  RUN(linear(f, "gemm_proj_ln", bw.proj, ws.outsc, f.N, p));
  TAP((tn + ".attn").c_str(), xout, 0, kC, f.N, kC);
  // ConvFFN (:39-46): fc1 + GELU
  base_params(p, bw.fc1);
  p.epi = EPI_STORE; p.act = ACT_GELU; p.n_real = kHid; p.out_bf16 = ws.H1; p.ldb = kHidp;
  RUN(linear(f, "gemm_fc1_gelu", bw.fc1, ws.xb0, f.N, p));
  }
  TAP((tn + ".fc1").c_str(), ws.H1, 1, kHidp, f.N, kHid);
  const bool need_shadow = (j == c.depths[i] - 1);      // the RHTB conv after the last block reads a bf16 shadow of the stream (:934)
  if (!h->simt && !h->direct_epilogue && !h->ffn_unfused) {
    // dwconv5 + GELU + input, fc2, norm2 and the residual add in one kernel: the hidden map h2 never reaches HBM
    // ... and, when another block of this layer follows, the casa statistics of the new stream for that block's window padding
    FfnStats fs; const FfnStats* fsp = nullptr;
    if (c.is_channel_spatial_attn && !need_shadow && !h->no_epilogue_stats) {
      const int wn = h->blocks[i][j + 1].win;
      fs = FfnStats{ws.cavg, ws.cmax, ws.part_sum, ws.part_max, round_up(f.band ? f.Hf : f.H, wn), round_up(f.W, wn)};
      fsp = &fs;
    }
    bf16* shadow = (need_shadow && fsp == nullptr) ? ws.xb0 : nullptr;      // emitted by the kernel's statistics warp
    FfnBand fb{2, f.row0, f.Hf};
    if (f.band != nullptr) RUN(fill_halo(f, ws.H1, (size_t)f.W * kHidp * sizeof(bf16), f.H, 2));   // the depthwise 5x5 reads two rows across the band edge
    LAUNCH("ffn_tail", 1, launch_ffn_tail(ws.H1, bw.dw_mma, bw.w2_img, bw.fc2.b, bw.g2, bw.b2, xout, f.B, f.H, f.W, fsp, shadow, h->num_sms, f.st,
                                          f.band ? &fb : nullptr));
    if (fsp != nullptr) f.stats_nparts = ffn_tiles_per_image(f.H, f.W);
    if (need_shadow && shadow == nullptr) LAUNCH("cast_shadow", 1, launch_cast_rows_bf16(xout, ws.xb0, f.N, f.st));
  } else {
#ifdef HITSIR_AB_PATHS
    LAUNCH("dwconv5", 1, launch_dwconv5_gelu_add(ws.H1, bw.dw_w, bw.dw_b, ws.H2, f.B, f.H, f.W, h->num_sms, f.st));
    // fc2 + norm2 + residual (:704)
    base_params(p, bw.fc2);
    p.epi = EPI_LN; p.n_real = kC; p.gamma = bw.g2; p.beta = bw.b2; p.res = xout; p.ldr = kC;
    p.out_f32 = xout; p.ldf = kC;
    if (need_shadow) { p.out_bf16 = ws.xb0; p.ldb = kCp; }
    RUN(linear(f, "gemm_fc2_ln", bw.fc2, ws.H2, f.N, p));
#else
    set_error("unfused FFN path is only available in the A/B test build (-DHITSIR_AB_PATHS)");
    return HITSIR_ERR_UNSUPPORTED;
#endif
  }
  TAP(tn.c_str(), xout, 0, kC, f.N, kC);
  return 0;
}

int union_attention(Fwd& f, int u, const float* a, const float* b, float* out) {
  // UnionAttention.forward (:113-133) on X = a (+ b)
  HitsirHandle* h = f.h;
  Workspace& ws = f.ws;
  LAUNCH("ua_stats", 2, launch_ua_stats(a, b, f.B, f.H, f.W, ws.cavg, ws.cmax, ws.havg, ws.hmax, ws.wavg, ws.wmax, f.st, f.band ? f.Hf : 0));
  if (f.band != nullptr) {
    // column statistics span the frame (all-reduce); the 3x3 convs over the (H, W) and (channel, H) planes read one row across the band edge
    RUN(band_allreduce(f, ws.havg, (int64_t)kC * f.W, ws.hmax, (int64_t)kC * f.W));
    RUN(fill_halo(f, ws.cavg, (size_t)f.W * sizeof(float), f.H, 1));
    RUN(fill_halo(f, ws.cmax, (size_t)f.W * sizeof(float), f.H, 1));
    RUN(fill_halo(f, ws.wavg, (size_t)kC * sizeof(float), f.H, 1));
    RUN(fill_halo(f, ws.wmax, (size_t)kC * sizeof(float), f.H, 1));
  }
  LAUNCH("ua_small", 1, launch_ua_small_convs(f.B, f.H, f.W, h->ua[u].small, ws.cavg, ws.cmax, ws.havg, ws.hmax, ws.wavg, ws.wmax, ws.c_att, ws.h_att, ws.w_att, f.st,
                                              f.top ? 1 : 0, f.bot ? 1 : 0));
  LAUNCH("ua_build", 1, launch_ua_build(f.B, f.H, f.W, ws.c_att, ws.h_att, ws.w_att, ws.outsc, f.st));
  GemmParams p;
  base_params(p, h->ua[u].conv_last);
  p.epi = EPI_STORE; p.n_real = kC; p.out_f32 = out; p.ldf = kC;
  return conv3(f, "conv_ua", h->ua[u].conv_last, ws.outsc, f.B, f.H, f.W, kCp, p);
}

// resi_connection='3conv' (:913-918, :1224-1231): out = conv3x3(C/4 -> C)(lrelu(conv1x1(lrelu(conv3x3(C -> C/4)(in))))) (+ res).
// The two C/4 = 45-channel maps live as bf16 [N, 64] in the (idle) self-correlation output buffer.
int resi_3conv(Fwd& f, int idx, const char* cat, const bf16* in, const float* res, float* out) {
  HitsirHandle* h = f.h;
  Workspace& ws = f.ws;
  const int C4 = kC / 4;
  bf16* t1 = ws.outsc;
  bf16* t2 = ws.outsc + f.Nl * 64;
  GemmParams p;
  base_params(p, h->r3_a[idx]);
  p.epi = EPI_STORE; p.act = ACT_LRELU; p.slope = 0.2f; p.n_real = C4; p.out_bf16 = t1; p.ldb = 64;
  RUN(conv3(f, cat, h->r3_a[idx], in, f.B, f.H, f.W, kCp, p));
  base_params(p, h->r3_b[idx]);
  p.epi = EPI_STORE; p.act = ACT_LRELU; p.slope = 0.2f; p.n_real = C4; p.out_bf16 = t2; p.ldb = 64;
  RUN(linear(f, cat, h->r3_b[idx], t1, f.N, p));
  base_params(p, h->r3_c[idx]);
  p.epi = EPI_STORE; p.n_real = kC; p.res = res; p.ldr = kC; p.out_f32 = out; p.ldf = kC;
  return conv3(f, cat, h->r3_c[idx], t2, f.B, f.H, f.W, 64, p);
}

int forward_impl(Fwd& f, const float* x, float* y) {
  HitsirHandle* h = f.h;
  const HitsirConfig& c = h->cfg;
  Workspace& ws = f.ws;
  const int B = f.B, H = f.H, W = f.W;
  const long long N = f.N;
  GemmParams p;
  // ---- mean shift + shallow features (:1310-1311, :1315/1322/1328/1337) + patch_embed LayerNorm (:975-983)
  bf16* A0 = ws.xb0;   // [N, first_kp <= 384] aliases xb0|xb1, dead before the second GEMM writes xb0
  LAUNCH("im2col", 1, launch_entry_im2col(x, A0, B, H, W, c.in_chans, h->first_f, h->first_kp, h->mean, c.img_range, f.st, f.row0, f.band ? f.Hf : 0));
  const float* pe_g = P(h, "patch_embed.norm.weight");
  const float* pe_b = P(h, "patch_embed.norm.bias");
  if (c.is_mult_size_conv_feat_extract) {
    bf16* G = ws.H1;   // [N,768] aliases H1|H2
    base_params(p, h->first);
    p.epi = EPI_MSGATE; p.n_real = kC; p.out_bf16 = G; p.ldb = 4 * kCp;
    RUN(linear(f, "gemm_first_msgate", h->first, A0, N, p));
    base_params(p, h->first_last);
    p.epi = EPI_STORE; p.n_real = kC; p.out_f32 = ws.S; p.ldf = kC;
    RUN(linear(f, "gemm_first_last", h->first_last, G, N, p));
  } else {
    base_params(p, h->first);
    p.epi = EPI_STORE; p.n_real = kC; p.out_f32 = ws.S; p.ldf = kC;
    RUN(linear(f, "gemm_first", h->first, A0, N, p));
  }
  // patch_embed LayerNorm (:975-983): shallow features S stay for the fusion, the stream starts from LN(S)
  if (c.ape_tokens > 0 && (long long)H * W != c.ape_tokens) {
    // x + absolute_pos_embed broadcasts (1, num_patches, C) against (B, H*W, C): any other size raises in the reference (:1294)
    set_error("The size of tensor a (%lld) must match the size of tensor b (%d) at non-singleton dimension 1 (absolute_pos_embed)", (long long)H * W, c.ape_tokens);
    return HITSIR_ERR_INVALID;
  }
  LAUNCH("ln_rows", 1, launch_ln_rows(ws.S, pe_g, pe_b, nullptr, ws.P, N, f.st, c.ape_tokens > 0 ? P(h, "absolute_pos_embed") : nullptr, c.ape_tokens));
  TAP("shallow", ws.S, 0, kC, N, kC);
  TAP("embed", ws.P, 0, kC, N, kC);
  // ---- deep features: RHTB stack (:1296-1297, :928-936)
  for (int i = 0; i < c.num_layers; ++i) {
    for (int j = 0; j < c.depths[i]; ++j) {
      RUN(forward_block(f, i, j, j == 0 ? ws.P : ws.Q, ws.Q));
      if (f.stopped) return 0;
    }
    if (c.resi_3conv) {
      RUN(resi_3conv(f, i, "conv_layer", ws.xb0, ws.P, ws.P));
    } else {
      base_params(p, h->layer_conv[i]);
      p.epi = EPI_STORE; p.n_real = kC; p.res = ws.P; p.ldr = kC; p.out_f32 = ws.P; p.ldf = kC;
      RUN(conv3(f, "conv_layer", h->layer_conv[i], ws.xb0, B, H, W, kCp, p));
    }
    TAP(("layer" + std::to_string(i)).c_str(), ws.P, 0, kC, N, kC);
  }
  // ---- final norm + conv_after_body (:1299-1300, :1317/1324/1330/1339)
  LAUNCH("ln_rows", 1, launch_ln_rows(ws.P, P(h, "norm.weight"), P(h, "norm.bias"), ws.xb0, nullptr, N, f.st));
  TAP("norm", ws.xb0, 1, kCp, N, kC);
  float* CAB = ws.Q;
  if (c.resi_3conv) {
    RUN(resi_3conv(f, c.num_layers, "conv_after_body", ws.xb0, nullptr, CAB));
  } else {
    base_params(p, h->conv_after_body);
    p.epi = EPI_STORE; p.n_real = kC; p.out_f32 = CAB; p.ldf = kC;
    RUN(conv3(f, "conv_after_body", h->conv_after_body, ws.xb0, B, H, W, kCp, p));
  }
  TAP("conv_after_body", CAB, 0, kC, N, kC);
  // ---- fusion(conv_after_body(deep), shallow): positional binding (:1330 -> :145)
  bf16* F = ws.xb1;
  if (c.is_fusion) {
    float* A1 = reinterpret_cast<float*>(ws.H1);       // [N,180] fp32 x2 inside H1|H2 (N*1536 B >= 2*N*720 B)
    float* A2 = A1 + N * kC;
    float* A3 = ws.P;                                  // the stream buffer is dead after the final norm
    RUN(union_attention(f, 0, CAB, nullptr, A1));
    RUN(union_attention(f, 1, CAB, ws.S, A2));
    RUN(union_attention(f, 2, ws.S, nullptr, A3));
    float* tapdst = (h->tap.dst != nullptr && h->tap.name == "fused") ? h->tap.dst : nullptr;
    if (tapdst != nullptr && N * kC > h->tap.floats) { set_error("tap 'fused' destination too small"); return HITSIR_ERR_INVALID; }
    LAUNCH("fusion_combine", 1, launch_fusion_combine(CAB, ws.S, A1, A2, A3, F, tapdst, N, f.st));
    if (tapdst != nullptr && h->tap.stop) { f.stopped = true; return 0; }
  } else {
    LAUNCH("fusion_add", 1, launch_add_to_bf16(CAB, ws.S, F, N, f.st));
    TAP("fused", F, 1, kCp, N, kC);
  }
  RUN(do_inject(f, "fused", nullptr, F, N));
  // ---- reconstruction (:1313-1340)
  const int s = c.upscale;
  const long long Nl = f.Nl;                                               // layout pixels (band mode: identical buffer offsets in every band)
  const size_t gap = f.band ? (size_t)2 * 4 * W * kNumFeat : 0;           // room for the halo rows of the upsampler maps
  auto last_params = [&](GemmParams& q, const GemmW& w, int ps) {
    base_params(q, w);
    q.epi = EPI_SHUFFLE_NCHW; q.ps = ps; q.n_real = c.in_chans * ps * ps; q.shuf_c = c.in_chans;
    q.out_scale = 1.0f / c.img_range;
    for (int k = 0; k < 4; ++k) q.mean[k] = h->mean[k];
    q.out_f32 = y;
  };
  if (c.upsampler == HITSIR_UP_NEAREST_CONV) {
    bf16* U0 = ws.up + gap;
    bf16* U1 = U0 + Nl * kNumFeat + gap;
    bf16* U2 = U1 + 4 * Nl * kNumFeat + gap;
    bf16* U3 = U2 + 16 * Nl * kNumFeat + gap;
    base_params(p, h->conv_before_upsample);
    p.epi = EPI_STORE; p.act = ACT_LRELU; p.slope = 0.01f; p.n_real = kNumFeat; p.out_bf16 = U0; p.ldb = kNumFeat;   // nn.LeakyReLU() default slope (:1251)
    RUN(conv3(f, "conv_before_upsample", h->conv_before_upsample, F, B, H, W, kCp, p));
    TAP("conv_before_upsample", U0, 1, kNumFeat, N, kNumFeat);
    // interpolate(x2, nearest) + conv_up{1,2} (:1331-1332) as sub-pixel convs on the map before the upsampling
    base_params(p, h->conv_up1);
    p.epi = EPI_STORE; p.act = ACT_LRELU; p.slope = 0.2f; p.n_real = kNumFeat; p.out_bf16 = U1; p.ldb = kNumFeat;
    RUN(conv3_up(f, "conv_up1", h->conv_up1, U0, B, H, W, p));
    TAP("up1", U1, 1, kNumFeat, 4 * N, kNumFeat);
    base_params(p, h->conv_up2);
    p.epi = EPI_STORE; p.act = ACT_LRELU; p.slope = 0.2f; p.n_real = kNumFeat; p.out_bf16 = U2; p.ldb = kNumFeat;
    RUN(conv3_up(f, "conv_up2", h->conv_up2, U1, B, 2 * H, 2 * W, p));
    TAP("up2", U2, 1, kNumFeat, 16 * N, kNumFeat);
    base_params(p, h->conv_hr);
    p.epi = EPI_STORE; p.act = ACT_LRELU; p.slope = 0.2f; p.n_real = kNumFeat; p.out_bf16 = U3; p.ldb = kNumFeat;
    RUN(conv3(f, "conv_hr", h->conv_hr, U2, B, 4 * H, 4 * W, kNumFeat, p));
    TAP("hr", U3, 1, kNumFeat, 16 * N, kNumFeat);
    last_params(p, h->conv_last, 1);
    RUN(conv3(f, "conv_last", h->conv_last, U3, B, 4 * H, 4 * W, kNumFeat, p));
  } else if (c.upsampler == HITSIR_UP_PIXELSHUFFLE) {
    bf16* U0 = ws.up + gap;
    bf16* Ua = U0 + Nl * kNumFeat + gap;
    bf16* Ub = Ua + 4 * Nl * kNumFeat + gap;
    base_params(p, h->conv_before_upsample);
    p.epi = EPI_STORE; p.act = ACT_LRELU; p.slope = 0.01f; p.n_real = kNumFeat; p.out_bf16 = U0; p.ldb = kNumFeat;
    RUN(conv3(f, "conv_before_upsample", h->conv_before_upsample, F, B, H, W, kCp, p));
    TAP("conv_before_upsample", U0, 1, kNumFeat, N, kNumFeat);
    const bf16* cur = U0;
    int ch = H, cw = W;
    if ((s & (s - 1)) == 0) {
      for (size_t k = 0; k < h->upsample.size(); ++k) {
        bf16* dst = (k % 2 == 0) ? Ua : Ub;
        if (k >= 2) { set_error("pixelshuffle upscale > 4 not supported by this build"); return HITSIR_ERR_UNSUPPORTED; }
        base_params(p, h->upsample[k]);
        p.epi = EPI_SHUFFLE_BF16; p.ps = 2; p.n_real = 4 * kNumFeat; p.shuf_c = kNumFeat; p.out_bf16 = dst; p.ldb = kNumFeat;
        RUN(conv3(f, "conv_pixelshuffle", h->upsample[k], cur, B, ch, cw, kNumFeat, p));
        cur = dst; ch *= 2; cw *= 2;
      }
    } else {
      base_params(p, h->upsample[0]);
      p.epi = EPI_SHUFFLE_BF16; p.ps = 3; p.n_real = 9 * kNumFeat; p.shuf_c = kNumFeat; p.out_bf16 = Ub; p.ldb = kNumFeat;
      RUN(conv3(f, "conv_pixelshuffle", h->upsample[0], cur, B, ch, cw, kNumFeat, p));
      cur = Ub; ch *= 3; cw *= 3;
    }
    last_params(p, h->conv_last, 1);
    RUN(conv3(f, "conv_last", h->conv_last, cur, B, ch, cw, kNumFeat, p));
  } else if (c.upsampler == HITSIR_UP_PIXELSHUFFLEDIRECT) {
    last_params(p, h->upsample[0], s);
    RUN(conv3(f, "conv_last_direct", h->upsample[0], F, B, H, W, kCp, p));
  } else {
    // upsampler=None / '' (:1335-1342): y = (x_shifted + conv_last(res)) / img_range + mean = x + conv_last(res) / img_range, same size as x
    last_params(p, h->conv_last, 1);
    p.res_img = x;
    RUN(conv3(f, "conv_last_none", h->conv_last, F, B, H, W, kCp, p));
  }
  return 0;
}

}  // namespace

// ==========================================================================================
// C ABI
// ==========================================================================================
extern "C" {

HITSIR_API const char* hitsir_last_error(void) { return g_err; }
HITSIR_API const char* hitsir_version(void) { return "hitsir_b200 0.1 (sm_100a, tcgen05+TMA)"; }

HITSIR_API int hitsir_create(const HitsirConfig* cfg, HitsirHandle** out) {
  if (!cfg || !out) { set_error("hitsir_create: null argument"); return HITSIR_ERR_INVALID; }
  *out = nullptr;
  int rc = validate_config(*cfg);
  if (rc) return rc;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) { set_error("hitsir_create: no CUDA device (%s); this library has no CPU path", cudaGetErrorString(e)); return HITSIR_ERR_CUDA; }
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, dev);
  if (e != cudaSuccess) { set_error("cudaGetDeviceProperties: %s", cudaGetErrorString(e)); return HITSIR_ERR_CUDA; }
  if (prop.major != 10) { set_error("hitsir_b200 needs an sm_100 (Blackwell B200) device, found sm_%d%d (%s)", prop.major, prop.minor, prop.name); return HITSIR_ERR_CUDA; }
  HitsirHandle* h = new HitsirHandle();
  h->cfg = *cfg;
  h->device = dev;
  h->num_sms = prop.multiProcessorCount;
  if (cfg->in_chans == 3) { h->mean[0] = 0.485f; h->mean[1] = 0.456f; h->mean[2] = 0.4060f; }   // (:1128)
#ifdef HITSIR_AB_PATHS
  const char* env = getenv("HITSIR_GEMM");
  h->simt = env && strcmp(env, "simt") == 0;
  const char* env5 = getenv("HITSIR_STATS");
  h->no_epilogue_stats = env5 && strcmp(env5, "kernel") == 0;
  const char* env7 = getenv("HITSIR_PROJFC1");
  h->projfc1_fused = env7 && strcmp(env7, "fused") == 0;
  const char* env8 = getenv("HITSIR_GEMMW");
  h->b_streamed = env8 && strcmp(env8, "streamed") == 0;
  const char* env4 = getenv("HITSIR_FFN");
  h->ffn_unfused = env4 && strcmp(env4, "unfused") == 0;
  const char* env3 = getenv("HITSIR_SCC");
  h->scc_gram_only = env3 && strcmp(env3, "gram") == 0;
  const char* env2 = getenv("HITSIR_EPILOGUE");
  h->direct_epilogue = env2 && strcmp(env2, "direct") == 0;
#endif
  build_param_list(h);
  e = cudaMalloc(reinterpret_cast<void**>(&h->arena), h->arena_floats * sizeof(float));
  if (e != cudaSuccess) { set_error("cudaMalloc(param arena): %s", cudaGetErrorString(e)); delete h; return HITSIR_ERR_CUDA; }
  *out = h;
  return 0;
}

HITSIR_API void hitsir_destroy(HitsirHandle* h) {
  if (!h) return;
  for (ProfRec& r : h->prof.recs) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
  for (cudaEvent_t e : h->prof.pool) cudaEventDestroy(e);
  free_owned(h);
  if (h->arena) cudaFree(h->arena);
  delete h;
}

HITSIR_API int hitsir_num_params(const HitsirHandle* h) { return h ? (int)h->params.size() : 0; }
HITSIR_API const char* hitsir_param_name(const HitsirHandle* h, int i) {
  if (!h || i < 0 || i >= (int)h->params.size()) return nullptr;
  return h->params[i].name.c_str();
}
HITSIR_API int64_t hitsir_param_numel(const HitsirHandle* h, int i) {
  if (!h || i < 0 || i >= (int)h->params.size()) return -1;
  return h->params[i].numel;
}

HITSIR_API int hitsir_set_param(HitsirHandle* h, const char* name, const float* data, int64_t numel, void* stream) {
  if (!h || !name || !data) { set_error("hitsir_set_param: null argument"); return HITSIR_ERR_INVALID; }
  auto it = h->index.find(name);
  if (it == h->index.end()) { set_error("Unexpected key(s) in state_dict: \"%s\"", name); return HITSIR_ERR_INVALID; }
  ParamSpec& p = h->params[it->second];
  if (p.numel != numel) { set_error("size mismatch for %s: expected %lld elements, got %lld", name, (long long)p.numel, (long long)numel); return HITSIR_ERR_INVALID; }
  HITSIR_CHECK(cudaMemcpyAsync(h->arena + p.offset, data, (size_t)numel * sizeof(float), cudaMemcpyDefault, (cudaStream_t)stream));
  p.set = true;
  h->finalized = false;
  return 0;
}

HITSIR_API int hitsir_finalize_weights(HitsirHandle* h, void* stream) {
  if (!h) { set_error("null handle"); return HITSIR_ERR_INVALID; }
  return finalize(h, (cudaStream_t)stream);
}

HITSIR_API int hitsir_workspace_bytes(const HitsirHandle* h, int B, int H, int W, size_t* bytes) {
  if (!h || !bytes || B < 1 || H < 1 || W < 1) { set_error("hitsir_workspace_bytes: bad argument"); return HITSIR_ERR_INVALID; }
  Workspace ws;
  int rc = layout_workspace(h, B, H, W, nullptr, &ws);
  if (rc) return rc;
  *bytes = ws.bytes;
  return 0;
}

HITSIR_API int hitsir_forward(HitsirHandle* h, const float* x, float* y, int B, int H, int W, void* workspace, size_t workspace_bytes, void* stream) {
  if (!h || !x || !y || !workspace) { set_error("hitsir_forward: null argument"); return HITSIR_ERR_INVALID; }
  if (!h->finalized) { set_error("hitsir_forward: weights not finalized (call hitsir_set_param for every key, then hitsir_finalize_weights)"); return HITSIR_ERR_WEIGHTS; }
  if ((long long)B * H * W * 16 >= 2147483647LL / 4) {
    // row indices are kept in 32 bit inside the GEMM tile maps; 16x upsampled pixel counts must fit too
    if ((long long)B * H * W * 16 >= 2147483647LL) { set_error("input too large: B*H*W*16 must be < 2^31"); return HITSIR_ERR_UNSUPPORTED; }
  }
  Fwd f;
  f.h = h; f.st = (cudaStream_t)stream; f.B = B; f.H = H; f.W = W; f.N = (long long)B * H * W; f.Nl = f.N;
  int rc = layout_workspace(h, B, H, W, workspace, &f.ws);
  if (rc) return rc;
  if (((uintptr_t)workspace & 255) != 0) { set_error("workspace must be 256-byte aligned"); return HITSIR_ERR_WORKSPACE; }
  if (f.ws.bytes > workspace_bytes) { set_error("workspace too small: need %zu bytes, got %zu", f.ws.bytes, workspace_bytes); return HITSIR_ERR_WORKSPACE; }
  h->launches = 0;
  rc = forward_impl(f, x, y);
  return rc;
}

HITSIR_API int hitsir_workspace_bytes_band(const HitsirHandle* h, int layout_h, int W, size_t* bytes) {
  if (!h || !bytes || layout_h < 1 || W < 1) { set_error("hitsir_workspace_bytes_band: bad argument"); return HITSIR_ERR_INVALID; }
  Workspace ws;
  int rc = layout_workspace(h, 1, layout_h, W, nullptr, &ws, 1);
  if (rc) return rc;
  *bytes = ws.bytes;
  return 0;
}

HITSIR_API int hitsir_forward_band(HitsirHandle* h, const float* x_frame, float* y_band, int H, int W, const HitsirBand* band, void* workspace,
                                   size_t workspace_bytes, void* stream) {
  if (!h || !x_frame || !y_band || !workspace || !band) { set_error("hitsir_forward_band: null argument"); return HITSIR_ERR_INVALID; }
  if (!h->finalized) { set_error("hitsir_forward_band: weights not finalized"); return HITSIR_ERR_WEIGHTS; }
  if ((band->has_top || band->has_bottom) && (!band->halo || !band->allreduce)) { set_error("hitsir_forward_band: exchange callbacks missing"); return HITSIR_ERR_INVALID; }
  if (H < 1 || H > band->layout_h || band->row0 < 0 || band->row0 + H > band->frame_h) { set_error("hitsir_forward_band: band rows [%d, %d) do not fit frame_h %d / layout_h %d", band->row0, band->row0 + H, band->frame_h, band->layout_h); return HITSIR_ERR_INVALID; }
  if (band->row0 % 192 != 0 || (band->has_bottom && H % 192 != 0)) {
    set_error("hitsir_forward_band: band boundaries must be multiples of 192 (lcm of the window sizes): row0 %d, rows %d", band->row0, H);
    return HITSIR_ERR_INVALID;
  }
  if (h->cfg.ape_tokens > 0) { set_error("hitsir_forward_band: ape=True is not supported in band mode"); return HITSIR_ERR_UNSUPPORTED; }
  if (h->cfg.upsampler == HITSIR_UP_NONE) { set_error("hitsir_forward_band: upsampler=None (same-size output added to the input) is not supported in band mode"); return HITSIR_ERR_UNSUPPORTED; }
  if (h->tap.dst != nullptr || h->inject.src != nullptr) { set_error("hitsir_forward_band: taps / injections are not supported in band mode"); return HITSIR_ERR_UNSUPPORTED; }
  Fwd f;
  f.h = h; f.st = (cudaStream_t)stream; f.B = 1; f.H = H; f.W = W; f.N = (long long)H * W; f.Nl = (long long)band->layout_h * W;
  f.band = band; f.ws_base = workspace; f.row0 = band->row0; f.Hf = band->frame_h; f.top = band->has_top != 0; f.bot = band->has_bottom != 0;
  int rc = layout_workspace(h, 1, band->layout_h, W, workspace, &f.ws, 1);
  if (rc) return rc;
  if (((uintptr_t)workspace & 255) != 0) { set_error("workspace must be 256-byte aligned"); return HITSIR_ERR_WORKSPACE; }
  if (f.ws.bytes > workspace_bytes) { set_error("workspace too small: need %zu bytes, got %zu", f.ws.bytes, workspace_bytes); return HITSIR_ERR_WORKSPACE; }
  // the reference pads the FRAME: a band of the last rows may be shorter than its own reflect padding only if the frame is
  for (int j = 0; j < h->cfg.depths[0]; ++j) {
    const int w = win_of(h->cfg, j), pad = round_up(H, w) - H;
    if (pad >= H) { set_error("band of %d rows is shorter than the reflect padding (%d) of window %d: merge it with its neighbour", H, pad, w); return HITSIR_ERR_INPUT_TOO_SMALL; }
  }
  h->launches = 0;
  return forward_impl(f, x_frame, y_band);
}

HITSIR_API int hitsir_forward_host(HitsirHandle* h, const float* host_x, float* host_y, int B, int H, int W, float* dev_x, float* dev_y,
                        void* workspace, size_t workspace_bytes, void* stream) {
  if (!h || !host_x || !host_y || !dev_x || !dev_y) { set_error("hitsir_forward_host: null argument"); return HITSIR_ERR_INVALID; }
  const size_t in_b = (size_t)B * h->cfg.in_chans * H * W * sizeof(float);
  const int se = h->cfg.upsampler == HITSIR_UP_NONE ? 1 : h->cfg.upscale;       // upsampler=None returns x-sized images whatever `upscale` says (:1344)
  const size_t out_b = in_b * se * se;
  HITSIR_CHECK(cudaMemcpyAsync(dev_x, host_x, in_b, cudaMemcpyHostToDevice, (cudaStream_t)stream));
  int rc = hitsir_forward(h, dev_x, dev_y, B, H, W, workspace, workspace_bytes, stream);
  if (rc) return rc;
  HITSIR_CHECK(cudaMemcpyAsync(host_y, dev_y, out_b, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  return 0;
}

HITSIR_API int hitsir_forward_u8(HitsirHandle* h, const uint8_t* x_hwc, uint8_t* y_hwc, int B, int H, int W, float* dev_x, float* dev_y,
                                 void* workspace, size_t workspace_bytes, void* stream) {
  if (!h || !x_hwc || !y_hwc || !dev_x || !dev_y) { set_error("hitsir_forward_u8: null argument"); return HITSIR_ERR_INVALID; }
  const int s = h->cfg.upsampler == HITSIR_UP_NONE ? 1 : h->cfg.upscale, ic = h->cfg.in_chans;
  if (launch_u8hwc_to_f32nchw(x_hwc, dev_x, B, H, W, ic, (cudaStream_t)stream)) return HITSIR_ERR_CUDA;
  int rc = hitsir_forward(h, dev_x, dev_y, B, H, W, workspace, workspace_bytes, stream);
  if (rc) return rc;
  if (launch_f32nchw_to_u8hwc(dev_y, y_hwc, B, H * s, W * s, ic, (cudaStream_t)stream)) return HITSIR_ERR_CUDA;
  h->launches += 2;
  return 0;
}

HITSIR_API int hitsir_f32nchw_to_u8hwc(const float* src, uint8_t* dst, int B, int C, int H, int W, void* stream) {
  if (!src || !dst || B <= 0 || C <= 0 || H <= 0 || W <= 0) { set_error("hitsir_f32nchw_to_u8hwc: bad argument"); return HITSIR_ERR_INVALID; }
  if (launch_f32nchw_to_u8hwc(src, dst, B, H, W, C, (cudaStream_t)stream)) return HITSIR_ERR_CUDA;
  return 0;
}

HITSIR_API int64_t hitsir_psnr_y_scratch_doubles(int B, int H, int W) {
  if (B <= 0 || H <= 0 || W <= 0) return 0;
  return (int64_t)B * psnr_y_chunks(H, W);
}

HITSIR_API int hitsir_psnr_y(const float* sr, const float* hr, int B, int H, int W, int clip_sr, double* scratch, double* mse_out, void* stream) {
  if (!sr || !hr || !scratch || !mse_out) { set_error("hitsir_psnr_y: null argument"); return HITSIR_ERR_INVALID; }
  if (B <= 0 || H <= 0 || W <= 0) { set_error("hitsir_psnr_y: bad shape %d x %d x %d", B, H, W); return HITSIR_ERR_INVALID; }
  if (launch_psnr_y(sr, hr, B, H, W, clip_sr, scratch, mse_out, (cudaStream_t)stream)) return HITSIR_ERR_CUDA;
  return 0;
}

HITSIR_API int hitsir_set_tap(HitsirHandle* h, const char* name, float* dst, int64_t dst_floats, int stop) {
  if (!h) { set_error("null handle"); return HITSIR_ERR_INVALID; }
  if (!name) { h->tap = Tap(); return 0; }
  h->tap.name = name; h->tap.dst = dst; h->tap.floats = dst_floats; h->tap.stop = stop;
  return 0;
}

HITSIR_API int hitsir_set_inject(HitsirHandle* h, const char* name, const float* src, int64_t src_floats) {
  if (!h) { set_error("null handle"); return HITSIR_ERR_INVALID; }
  if (!name) { h->inject = Inject(); return 0; }
  if (!src) { set_error("hitsir_set_inject: null source"); return HITSIR_ERR_INVALID; }
  h->inject.name = name; h->inject.src = src; h->inject.floats = src_floats;
  return 0;
}

HITSIR_API int hitsir_get_bias_table(HitsirHandle* h, int layer, int block, float* dst, int64_t dst_floats, void* stream) {
  if (!h || !dst) { set_error("hitsir_get_bias_table: null argument"); return HITSIR_ERR_INVALID; }
  if (!h->finalized) { set_error("hitsir_get_bias_table: weights not finalized"); return HITSIR_ERR_WEIGHTS; }
  if (layer < 0 || layer >= (int)h->blocks.size() || block < 0 || block >= (int)h->blocks[layer].size()) {
    set_error("hitsir_get_bias_table: no block %d.%d", layer, block); return HITSIR_ERR_INVALID;
  }
  const BlockW& bw = h->blocks[layer][block];
  const int64_t n = (int64_t)kHeads * bw.win * bw.win * bw.base * bw.base;
  if (dst_floats != n) { set_error("hitsir_get_bias_table: block %d.%d has %lld values (6 x L x Lb), destination %lld", layer, block, (long long)n, (long long)dst_floats); return HITSIR_ERR_INVALID; }
  HITSIR_CHECK(cudaMemcpyAsync(dst, bw.bias_tbl, (size_t)n * sizeof(float), cudaMemcpyDefault, (cudaStream_t)stream));
  return 0;
}

HITSIR_API int64_t hitsir_last_launch_count(const HitsirHandle* h) { return h ? h->launches : 0; }

HITSIR_API int hitsir_profile_enable(HitsirHandle* h, int on) {
  if (!h) { set_error("null handle"); return HITSIR_ERR_INVALID; }
  h->prof.on = on != 0;
  for (ProfRec& r : h->prof.recs) { h->prof.pool.push_back(r.a); h->prof.pool.push_back(r.b); }
  h->prof.recs.clear();
  return 0;
}
HITSIR_API int hitsir_profile_num_categories(const HitsirHandle* h) { return h ? (int)h->prof.cats.size() : 0; }
HITSIR_API int hitsir_profile_get(HitsirHandle* h, int i, const char** name, double* total_ms, int64_t* launches) {
  if (!h || i < 0 || i >= (int)h->prof.cats.size()) { set_error("hitsir_profile_get: bad index"); return HITSIR_ERR_INVALID; }
  double ms = 0.0; int64_t n = 0;
  for (const ProfRec& r : h->prof.recs) {
    if (r.cat != i) continue;
    float t = 0.f;
    HITSIR_CHECK(cudaEventElapsedTime(&t, r.a, r.b));
    ms += t; ++n;
  }
  *name = h->prof.cats[i].c_str(); *total_ms = ms; *launches = n;
  return 0;
}

HITSIR_API int hitsir_set_gemm_backend(HitsirHandle* h, const char* backend) {
  if (!h || !backend) { set_error("null argument"); return HITSIR_ERR_INVALID; }
  if (strcmp(backend, "umma") == 0) { h->simt = false; h->direct_epilogue = false; }
#ifdef HITSIR_AB_PATHS
  // the direct-store epilogues need the unfused FFN tail, which only this build compiles
  else if (strcmp(backend, "umma_direct") == 0) { h->simt = false; h->direct_epilogue = true; }
  else if (strcmp(backend, "simt") == 0) h->simt = true;
#endif
  else { set_error("unknown gemm backend '%s' (umma; 'umma_direct' and 'simt' only in the -DHITSIR_AB_PATHS test build)", backend); return HITSIR_ERR_INVALID; }
  return 0;
}

}  // extern "C"
