// Y channel of YCbCr as the reference evaluation computes it, shared by the metrics on the device (psnr_y and ssim_y in
// metrics.cu): utils/utils.py:170-186 writes 16/255 + (65.738 R + 129.057 G + 25.064 B) / 256, every operation rounded to fp32 in that
// order (no FMA contraction).
#pragma once
#include <cuda_runtime.h>

namespace hitsir {

__device__ __forceinline__ float y_channel(float r, float g, float b) {
  const float t = __fadd_rn(__fadd_rn(__fmul_rn(65.738f, r), __fmul_rn(129.057f, g)), __fmul_rn(25.064f, b));
  return __fadd_rn((float)(16.0 / 255.0), __fdiv_rn(t, 256.0f));
}

// Y of a uint8 RGB pixel as BasicSR 1.4.2 scores it (basicsr/metrics/metric_util.py to_y_channel, bgr2ycbcr of
// basicsr/utils/color_util.py), on the 0-255 scale: t = fp32(v) / 255 in fp32; y = ((24.966 t_b + 128.553 t_g) + 65.481 t_r) + 16 in
// double (numpy's dot of a float32 BGR pixel with the float64 coefficients); fp32(y / 255); then * 255 in fp32.  Every operation is
// an explicit _rn intrinsic so that no contraction changes a value: equal to numpy for all 2^24 triples (tested on the CPU).
__device__ __forceinline__ float y_basicsr(unsigned r, unsigned g, unsigned b) {
  const double tr = (double)__fdiv_rn((float)r, 255.f), tg = (double)__fdiv_rn((float)g, 255.f), tb = (double)__fdiv_rn((float)b, 255.f);
  const double y = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(24.966, tb), __dmul_rn(128.553, tg)), __dmul_rn(65.481, tr)), 16.0);
  return __fmul_rn(__double2float_rn(__ddiv_rn(y, 255.0)), 255.f);
}

}  // namespace hitsir
