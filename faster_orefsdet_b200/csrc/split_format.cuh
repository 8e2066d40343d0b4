// The fp16 split operand format of the tensor-core kernels.  An fp32 operand x is scaled by a power of two 2^e that puts
// the largest magnitude of the tensor into [2^13, 2^14) and stored as hi = fp16(x * 2^e), lo = fp16(x * 2^e - hi)
// (22 significant bits); the MMAs form hi.hi + lo.hi + hi.lo.  In memory, per pixel and per 16 channels, one 64-byte
// group [16 x fp16 hi | 16 x fp16 lo].  A producer that writes this format publishes the bound it took 2^e from, and the
// consumer derives the same 2^e from that bound with pow2_scale: both sides must use this one rule, bit for bit.
#pragma once
#include <cuda_fp16.h>
#include <stdint.h>

namespace fod {

// 2^e with amax * 2^e in [2^13, 2^14) (and its inverse); 1 for zero / denormal-range / non-finite bounds
__device__ __forceinline__ void pow2_scale(float amax, float& scale, float& inv) {
  const int E = (int)((__float_as_uint(amax) >> 23) & 0xFF);
  if (E < 32 || E > 240) {
    scale = 1.f;
    inv = 1.f;
  } else {
    scale = __uint_as_float((uint32_t)(267 - E) << 23);  // 2^(13 - (E - 127))
    inv = __uint_as_float((uint32_t)(E - 13) << 23);
  }
}

// (a, b) -> packed fp16 pair of the rounded values (a in the low half) and of the exact remainders
__device__ __forceinline__ void split_f16x2(float a, float b, uint32_t& hi, uint32_t& lo) {
  const __half2 h = __floats2half2_rn(a, b);
  const float2 hf = __half22float2(h);
  const __half2 l = __floats2half2_rn(a - hf.x, b - hf.y);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}

}  // namespace fod
