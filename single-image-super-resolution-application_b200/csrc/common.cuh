// Shared device/host helpers for the hitsir_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda.h>
#include <stdint.h>
#include <stdio.h>

#define HITSIR_CHECK(expr)                                                              \
  do {                                                                                  \
    cudaError_t _e = (expr);                                                            \
    if (_e != cudaSuccess) {                                                            \
      hitsir::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return 1;                                                                         \
    }                                                                                   \
  } while (0)

namespace hitsir {

typedef __nv_bfloat16 bf16;

void set_error(const char* fmt, ...);

// Opt a kernel in to its dynamic shared-memory size once per (kernel, device): the attribute is per device, and a process may
// drive several (the per-call `mask` static lives at the call site, one per kernel instantiation).
template <class Kernel>
static inline int ensure_dynamic_smem(Kernel kernel, int bytes, unsigned long long* mask) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) { set_error("cudaGetDevice failed"); return 1; }
  const unsigned long long bit = 1ull << (dev & 63);
  if (*mask & bit) return 0;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e != cudaSuccess) { set_error("cudaFuncSetAttribute(MaxDynamicSharedMemorySize=%d) -> %s", bytes, cudaGetErrorString(e)); return 1; }
  *mask |= bit;
  return 0;
}

static inline int cdiv(int a, int b) { return (a + b - 1) / b; }
static inline int64_t cdiv64(int64_t a, int64_t b) { return (a + b - 1) / b; }
static inline int round_up(int a, int b) { return cdiv(a, b) * b; }

// ---------------------------------------------------------------------------
// small math
// ---------------------------------------------------------------------------
__device__ __forceinline__ float ex2_approx(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_approx(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float tanh_approx(float x) { float y; asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
// Packed-fp32 GELU (erf form, hit_sir_pro.py:32 nn.GELU) for two values: x * Phi(x) with
// Phi(x) ~= 1 / (1 + 2^(-x (a + b s + c s^2))), s = min(x^2, 81): a minimax fit of the normal CDF by a logistic of an odd quintic
// (|error| <= 1.6e-5 * max(|x|, 1) evaluated in fp32 with ex2.approx / rcp.approx; the quintic turns over at |x| ~ 11.4, beyond 9 the logistic
// is saturated anyway).  The logistic is written with ONE MUFU op per value: 1 / (1 + 2^z) = (1 + tanh(-z ln2 / 2)) / 2, so
// x Phi(x) = hx + hx tanh(w) with hx = x / 2, w = x (a' + b' s + c' s^2) (the quintic scaled by ln2 / 2).  5 packed FMA-pipe instructions + 2 FMNMX + 2 MUFU per pair, against 6 + 2 + 4 for
// the ex2 + rcp form and 12 + 4 FMNMX for a polynomial-only form: the FMA pipe is the binding resource of the FFN kernels, and the fc1
// epilogue was MUFU-bound with the ex2 + rcp form (67 % of the pipe, profiles/r1i).  tanh.approx.f32 has a relative error of 2^-11, i.e. an
// ABSOLUTE error of up to 2.4e-4 |x| on the result (where x < 0 the result itself is smaller than that) -- an eighth of the bf16 rounding step
// of a stored value of magnitude |x|, which is what the consumers of h1 / h2 see anyway.
__device__ __forceinline__ float2 gelu2(float2 x) {
  float2 s = __fmul2_rn(x, x);
  s.x = fminf(s.x, 81.f); s.y = fminf(s.y, 81.f);
  float2 p = __ffma2_rn(s, make_float2(-3.286197700e-04f, -3.286197700e-04f), make_float2(3.687881087e-02f, 3.687881087e-02f));
  p = __ffma2_rn(p, s, make_float2(7.976246503e-01f, 7.976246503e-01f));
  const float2 w = __fmul2_rn(p, x);
  const float2 hx = __fmul2_rn(x, make_float2(0.5f, 0.5f));
  return __ffma2_rn(hx, make_float2(tanh_approx(w.x), tanh_approx(w.y)), hx);
}

__device__ __forceinline__ float lrelu(float x, float slope) { return x > 0.f ? x : x * slope; }
__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + __expf(-x)); }

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float2 unpack_bf16x2(uint32_t u) {
  __nv_bfloat162 v = *reinterpret_cast<__nv_bfloat162*>(&u);
  return __bfloat1622float2(v);
}
// bf16 pair -> fp32 pair with two byte permutes: keeps the conversion on the ALU pipe (the compiler's own choice puts every other one on
// the FMA pipe as IMAD.U32 x 65536, which is the saturated pipe of the depthwise-conv loops)
__device__ __forceinline__ float2 unpack_bf16x2_alu(uint32_t u) {
  uint32_t lo, hi;
  asm("prmt.b32 %0, %1, 0, 0x1044;" : "=r"(lo) : "r"(u));
  asm("prmt.b32 %0, %1, 0, 0x3244;" : "=r"(hi) : "r"(u));
  return make_float2(__uint_as_float(lo), __uint_as_float(hi));
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ---------------------------------------------------------------------------
// PTX wrappers: mbarrier, TMA, tcgen05 (Blackwell sm_100a)
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// one arrival per warp: every lane has finished (and fenced) its writes, lane 0 signals for the whole warp
__device__ __forceinline__ void mbar_arrive_warp(uint32_t bar) {
  __syncwarp();
  if ((threadIdx.x & 31) == 0) mbar_arrive(bar);
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "LAB_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra DONE;\n\t"
      "bra LAB_WAIT;\n\t"
      "DONE:\n\t"
      "}" ::"r"(bar), "r"(parity) : "memory");
}
// Same wait for the single-role warps (producer, MMA issuer, DMA, statistics) that share a scheduler with four compute warps: the plain
// loop above re-issues try_wait every ~7 cycles (ncu: a third of all instructions of ffn_tail were SYNCS / BRA / YIELD of role warps,
// 43 % of the issue slots of the sub-partition that hosts the statistics warp).  With a suspend-time hint the hardware parks the
// thread until the phase completes (or the hint expires) instead of returning at once.
__device__ __forceinline__ void mbar_wait_park(uint32_t bar, uint32_t parity, uint32_t hint_ns = 1000u) {
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "LAB_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1, %2;\n\t"
      "@P1 bra DONE;\n\t"
      "bra LAB_WAIT;\n\t"
      "DONE:\n\t"
      "}" ::"r"(bar), "r"(parity), "r"(hint_ns) : "memory");
}
// mbarrier wait with a watchdog: a protocol bug traps (-> launch error) instead of hanging the device
__device__ __forceinline__ void wait_bar(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  long long spins = 0;
  while (true) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    if (done) break;
    if (++spins > (1LL << 26)) {
      printf("mbarrier timeout (block %d thread %d bar %u parity %u)\n", blockIdx.x, threadIdx.x, (bar >> 3) & 31u, parity);
      __trap();
    }
  }
}
// barrier `id` (1..15) over the first `nthreads` threads that reach it: a subset of the CTA's warps synchronises without the others
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }
// Programmatic dependent launch (the per-block chain casa gate -> SCC -> proj -> fc1 -> FFN tail -> pool MLP is 6 dependent launches x 36
// blocks; on small inputs the grid launch latency between them is a sixth of the forward).  A kernel launched with launch_pdl() may
// become resident while its predecessor in the stream is still draining; pdl_entry() holds it until that grid has completed and its
// writes are visible, then lets the NEXT launch in the stream do the same.  Everything before pdl_entry() may only touch memory that no
// kernel of the forward writes (weights, shared memory, TMEM, barriers).  Kernels launched without the attribute see a no-op.
__device__ __forceinline__ void pdl_entry() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
template <class... KArgs, class... Args>
static inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(tmap) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const void* tmap, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(tmap), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
// one contiguous block global -> shared through the bulk-copy engine (size and both addresses multiples of 16 bytes)
__device__ __forceinline__ void bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const void* tmap, uint32_t bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(tmap), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
// shared -> global tensor stores, tracked as bulk groups of the issuing thread
__device__ __forceinline__ void tma_store_2d(const void* tmap, uint32_t src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(tmap), "r"(src), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_store_4d(const void* tmap, uint32_t src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(tmap), "r"(src), "r"(c0), "r"(c1),
               "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// until at most N of this thread's bulk groups are still reading shared memory (N = 1: all but the newest)
template <int N>
__device__ __forceinline__ void tma_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
// until every bulk group of this thread has completed (its global writes done)
__device__ __forceinline__ void tma_wait_all0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]; bf16 inputs, fp32 accumulate
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// arrive on an mbarrier once all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// 32 lanes x 16 consecutive fp32 columns: thread i of the warp receives lane (base_lane + i)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// Batched form: issue several tmem_ld16_nw, then ONE tmem_ld_wait, then reg_fence16 on every destination group (ties the registers to
// a point after the wait so the compiler cannot hoist their uses above it).
__device__ __forceinline__ void tmem_ld16_nw(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void reg_fence16(uint32_t* r) {
  asm volatile("" : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                    "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]));
}

// NG x 16 consecutive accumulator columns of this thread's TMEM lane -> registers with a single wait
template <int NG>
__device__ __forceinline__ void tmem_ld_cols(uint32_t taddr, float (&v)[NG][16]) {
  uint32_t r[NG][16];
#pragma unroll
  for (int i = 0; i < NG; ++i) tmem_ld16_nw(taddr + 16 * i, r[i]);
  tmem_ld_wait();
#pragma unroll
  for (int i = 0; i < NG; ++i) {
    reg_fence16(r[i]);
#pragma unroll
    for (int e = 0; e < 16; ++e) v[i][e] = __uint_as_float(r[i][e]);
  }
}
// 32 consecutive fp32 columns with a single wait (the same loads as tmem_ld_cols<2>; written out, it keeps the conv3_c64_up epilogue's
// instruction schedule)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
  uint32_t r0[16], r1[16];
  tmem_ld16_nw(taddr, r0);
  tmem_ld16_nw(taddr + 16, r1);
  tmem_ld_wait();
  reg_fence16(r0);
  reg_fence16(r1);
#pragma unroll
  for (int i = 0; i < 16; ++i) { v[i] = __uint_as_float(r0[i]); v[16 + i] = __uint_as_float(r1[i]); }
}

// 16-byte chunk address inside a SWIZZLE_128B block with 128-byte rows
__device__ __forceinline__ uint8_t* swz(uint8_t* block, int row, int chunk) { return block + row * 128 + ((chunk ^ (row & 7)) << 4); }
// 16 fp32 values -> bf16 chunks chunk0, chunk0 + 1 of `row`
__device__ __forceinline__ void store16(uint8_t* block, int row, int chunk0, const float* v) {
  *reinterpret_cast<uint4*>(swz(block, row, chunk0)) =
      make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
  *reinterpret_cast<uint4*>(swz(block, row, chunk0 + 1)) =
      make_uint4(pack_bf16x2(v[8], v[9]), pack_bf16x2(v[10], v[11]), pack_bf16x2(v[12], v[13]), pack_bf16x2(v[14], v[15]));
}

// UMMA shared-memory matrix descriptor, SWIZZLE_128B (layout type 2), descriptor version 1 (sm_100).  K-major: lbo ignored, sbo = 1024
// (8 rows of 128 B).  MN-major: lbo = stride between 64-element blocks along M/N, sbo = stride between 8-row groups along K
// (cute/atom/mma_traits_sm100.hpp canonical forms).
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);      // start address, bits [0,14)
  d |= (uint64_t)(lbo_bytes >> 4) << 16;         // bits [16,30)
  d |= (uint64_t)(sbo_bytes >> 4) << 32;         // bits [32,46)
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// K-major operand with 128-byte rows
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) { return make_desc(saddr, 16, 1024); }
// instruction descriptor for kind::f16: D = f32, A = B = bf16, M = m, N = n; a_mn / b_mn = 1: that operand is MN-major (0: K-major)
__host__ __device__ constexpr uint32_t make_idesc(int m, int n, int a_mn, int b_mn) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) | ((uint32_t)(n >> 3) << 17) |
         ((uint32_t)(m >> 4) << 24);
}
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int m, int n) { return make_idesc(m, n, 0, 0); }

// warp-level bf16 MMA m16n8k16, fp32 accumulate in place: A = four fragment registers, B = two
__device__ __forceinline__ void mma_bf16_16816(float* d, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3]) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

}  // namespace hitsir
