// Y channel of YCbCr as the reference evaluation computes it, shared by the metrics on the device (psnr_y in glue.cu, ssim_y in
// ssim.cu): utils/utils.py:170-186 writes 16/255 + (65.738 R + 129.057 G + 25.064 B) / 256, every operation rounded to fp32 in that
// order (no FMA contraction).
#pragma once
#include <cuda_runtime.h>

namespace hitsir {

__device__ __forceinline__ float y_channel(float r, float g, float b) {
  const float t = __fadd_rn(__fadd_rn(__fmul_rn(65.738f, r), __fmul_rn(129.057f, g)), __fmul_rn(25.064f, b));
  return __fadd_rn((float)(16.0 / 255.0), __fdiv_rn(t, 256.0f));
}

}  // namespace hitsir
