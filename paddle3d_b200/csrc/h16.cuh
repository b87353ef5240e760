// The fp16-pair ("H16") encoding of the tensor-core paths: x = hi + lo' * 2^-11, with hi = fp16(x) and
// lo' = fp16((x - hi) * 2^11).  Every kernel that writes or reads pair rows or pixel images uses these helpers, so the
// encoding is defined once.
#pragma once
#include <cuda_fp16.h>

namespace p3d {

constexpr float kLoScale = 2048.0f, kLoInv = 1.0f / 2048.0f;

// x -> (hi, lo') fp16 pair; sets ovf when |x| leaves fp16's range (value saturated to +-65504)
__device__ __forceinline__ void split_h16(float x, __half &hi, __half &lo, bool &ovf) {
  if (fabsf(x) > 65504.0f) {
    ovf = true;
    x = copysignf(65504.0f, x);
  }
  hi = __float2half_rn(x);
  lo = __float2half_rn((x - __half2float(hi)) * kLoScale);
}
__device__ __forceinline__ float merge_h16(__half hi, __half lo) { return fmaf(__half2float(lo), kLoInv, __half2float(hi)); }

}  // namespace p3d
