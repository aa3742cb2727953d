// Half-precision edge of the offline Hankel-4 kernels: fp16 / bf16 signals and sub-bands are widened to fp32 exactly in the loads
// and the fp32 results are rounded to nearest even in the stores.  Everything between (the two-term fp16 split of the operands, the
// MMAs, the fp32 accumulation) is the fp32 instantiation's, so a half-precision call is bit-identical to the fp32 call on the
// widened input followed by a round-to-nearest-even cast of its output.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

namespace pqmf {

// sample format of a Hankel-4 instantiation's input and output (the bank and the accumulation are always the same)
enum class H4Io : int {
  F32 = 0,   // float32 rows / sub-bands
  F16 = 1,   // IEEE half rows / sub-bands
  BF16 = 2,  // bfloat16 rows / sub-bands
  PCM = 3,   // int16 WAV frames in (analysis) or out (synthesis), float32 sub-bands (pcm.cuh)
};
__host__ __device__ constexpr bool h4_io_half(H4Io io) { return io == H4Io::F16 || io == H4Io::BF16; }

// two packed half words -> two floats (exact: every fp16 and bf16 value is an fp32 value)
template <H4Io IO>
__device__ __forceinline__ float2 h4_widen2(uint32_t w) {
  if constexpr (IO == H4Io::F16) {
    __half2 h;
    memcpy(&h, &w, 4);
    return __half22float2(h);
  } else {
    // bf16 is the upper half of an fp32 word
    return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xFFFF0000u));
  }
}
// two floats -> two packed half words, each rounded to nearest even (what torch's .to(torch.float16 / bfloat16) does)
template <H4Io IO>
__device__ __forceinline__ uint32_t h4_narrow2(float a, float b) {
  uint32_t w;
  if constexpr (IO == H4Io::F16) {
    const __half2 h = __floats2half2_rn(a, b);
    memcpy(&w, &h, 4);
  } else {
    const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    memcpy(&w, &h, 4);
  }
  return w;
}
template <H4Io IO>
__device__ __forceinline__ uint16_t h4_narrow1(float a) {
  uint16_t u;
  if constexpr (IO == H4Io::F16) {
    const __half h = __float2half_rn(a);
    memcpy(&u, &h, 2);
  } else {
    const __nv_bfloat16 h = __float2bfloat16_rn(a);
    memcpy(&u, &h, 2);
  }
  return u;
}

// eight consecutive half samples held as four raw words in v[0..3] (one 16-byte load) -> eight floats in v[0..7]
template <H4Io IO>
__device__ __forceinline__ void h4_widen8(float (&v)[8]) {
  const uint32_t w[4] = {__float_as_uint(v[0]), __float_as_uint(v[1]), __float_as_uint(v[2]), __float_as_uint(v[3])};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 f = h4_widen2<IO>(w[i]);
    v[2 * i] = f.x;
    v[2 * i + 1] = f.y;
  }
}
// four consecutive half frames held as two raw words in .x / .y (one 8-byte load) -> four floats
template <H4Io IO>
__device__ __forceinline__ float4 h4_widen4(const float4& raw) {
  const float2 lo = h4_widen2<IO>(__float_as_uint(raw.x)), hi = h4_widen2<IO>(__float_as_uint(raw.y));
  return make_float4(lo.x, lo.y, hi.x, hi.y);
}

}  // namespace pqmf
