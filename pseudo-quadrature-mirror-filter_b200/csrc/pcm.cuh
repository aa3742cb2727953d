// int16 PCM edge of the PQMF path (SURVEY 8f-4): de-interleave + int16 -> fp32 fused into the analysis loads, fp32 -> int16 +
// interleave fused into the synthesis stores.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace pqmf {

// ---- int16 PCM edge (SURVEY 8f-4).  WAV frames are interleaved [clip][time][channel]; torchaudio.load turns them into
//      float32 / 32768 per channel (what every wrapper of the reference feeds the PQMF: PQMFWrapper.py:113,
//      1-PitchShifterWrapper.py:348) and PitchShifterPvoc/2-TestBlocks.py:26-30 down-mixes with mean(dim=0). ----
struct PcmIn {
  const int16_t* pcm;  // [clips, T, C] or nullptr (fp32 rows)
  int C;               // channels per WAV frame
  int downmix;         // 1: one row per clip = mean over the channels (fp32 sum in channel order, then / C, as torch.mean does)
};
// sample s of row b (row = clip * C + channel, or clip when down-mixing); T = frames per clip
__device__ __forceinline__ float pcm_sample(const PcmIn& in, long b, long s, long T) {
  constexpr float kInv = 1.0f / 32768.0f;
  if (in.downmix) {
    const int16_t* f = in.pcm + ((size_t)b * T + s) * in.C;
    float acc = 0.f;
    for (int c = 0; c < in.C; ++c) acc += (float)f[c] * kInv;
    return acc / (float)in.C;
  }
  const long clip = b / in.C;
  const int ch = (int)(b - clip * in.C);
  return (float)in.pcm[((size_t)clip * T + s) * in.C + ch] * kInv;
}
// fp32 -> PCM: round to nearest even, saturate (torch: clamp(round(v * 32768), -32768, 32767).to(int16))
__device__ __forceinline__ int16_t pcm_quantise(float v) {
  const float q = rintf(v * 32768.0f);
  return (int16_t)(q < -32768.f ? -32768.f : (q > 32767.f ? 32767.f : q));
}

// both int16 halves of a 32-bit word as float / 32768, exactly, without I2F: XOR the sign bits (offset binary u = v + 32768), drop each
// half into the mantissa of 2^23 (PRMT), and one FMA maps 2^23 + u to (u - 32768) / 32768
__device__ __forceinline__ void pcm_pair(int word, float& lo, float& hi) {
  const uint32_t w = (uint32_t)word ^ 0x80008000u;
  lo = fmaf(__uint_as_float(__byte_perm(w, 0x4B000000u, 0x7610)), 1.0f / 32768.0f, -257.0f);
  hi = fmaf(__uint_as_float(__byte_perm(w, 0x4B000000u, 0x7632)), 1.0f / 32768.0f, -257.0f);
}

// eight consecutive samples s .. s + 7 of row b (s a multiple of 8, T a multiple of 8), in two steps so that a kernel can keep the RAW
// words in registers across its prefetch distance and convert when it consumes them: pcm_load8_raw issues one 16-byte load for mono,
// one 32-byte load for stereo (either channel or the down-mix) and converts on the spot only beyond two channels (element-wise loads);
// pcm_convert8 turns the raw words into floats / 32768.
__device__ __forceinline__ void pcm_load8_raw(const PcmIn& in, long b, long s, long T, float (&v)[8]) {
  if (in.C == 1) {
    const int4 raw = __ldg(reinterpret_cast<const int4*>(in.pcm + (size_t)b * T + s));
    v[0] = __int_as_float(raw.x); v[1] = __int_as_float(raw.y); v[2] = __int_as_float(raw.z); v[3] = __int_as_float(raw.w);
  } else if (in.C == 2) {
    const long clip = in.downmix ? b : (b >> 1);
    const int4* src = reinterpret_cast<const int4*>(in.pcm + ((size_t)clip * T + s) * 2);
    const int4 r0 = __ldg(src), r1 = __ldg(src + 1);
    v[0] = __int_as_float(r0.x); v[1] = __int_as_float(r0.y); v[2] = __int_as_float(r0.z); v[3] = __int_as_float(r0.w);
    v[4] = __int_as_float(r1.x); v[5] = __int_as_float(r1.y); v[6] = __int_as_float(r1.z); v[7] = __int_as_float(r1.w);
  } else {
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = pcm_sample(in, b, s + i, T);
  }
}
__device__ __forceinline__ void pcm_convert8(const PcmIn& in, long b, float (&v)[8]) {
  if (in.C == 1) {
    const int w[4] = {__float_as_int(v[0]), __float_as_int(v[1]), __float_as_int(v[2]), __float_as_int(v[3])};
#pragma unroll
    for (int i = 0; i < 4; ++i) pcm_pair(w[i], v[2 * i], v[2 * i + 1]);
  } else if (in.C == 2) {
    const int ch = in.downmix ? 0 : (int)(b & 1);
#pragma unroll
    for (int i = 0; i < 8; ++i) {  // one WAV frame (left, right) per word
      float l, r;
      pcm_pair(__float_as_int(v[i]), l, r);
      v[i] = in.downmix ? (l + r) / 2.0f : (ch ? r : l);
    }
  }
}

// pcm_load8_raw for the streaming kernels, whose rows and blocks stay below 2^31 (32-bit index arithmetic): the same 16-byte mono and
// 32-byte stereo loads (raw words for pcm_convert8), and for more channels one pass over each frame's channels, converted on the spot
// (pcm_sample's arithmetic: the down-mix sums in channel order, then divides by C)
__device__ __forceinline__ void pcm_load8_raw_row(const PcmIn& in, int b, int s, int T, float (&v)[8]) {
  int4 r0, r1;
  if (in.C == 1) {
    r0 = __ldg(reinterpret_cast<const int4*>(in.pcm + (size_t)b * T + s));
    r1 = make_int4(0, 0, 0, 0);
  } else if (in.C == 2) {
    const int4* src = reinterpret_cast<const int4*>(in.pcm + ((size_t)(in.downmix ? b : (b >> 1)) * T + s) * 2);
    r0 = __ldg(src);
    r1 = __ldg(src + 1);
  } else {
    constexpr float kInv = 1.0f / 32768.0f;
    const int clip = in.downmix ? b : b / in.C;
    const int16_t* f = in.pcm + ((size_t)clip * T + s) * in.C + (in.downmix ? 0 : b - clip * in.C);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (in.downmix) {
        float acc = 0.f;
        for (int c = 0; c < in.C; ++c) acc += (float)__ldg(f + i * in.C + c) * kInv;
        v[i] = acc / (float)in.C;
      } else {
        v[i] = (float)__ldg(f + i * in.C) * kInv;
      }
    }
    return;
  }
  v[0] = __int_as_float(r0.x); v[1] = __int_as_float(r0.y); v[2] = __int_as_float(r0.z); v[3] = __int_as_float(r0.w);
  v[4] = __int_as_float(r1.x); v[5] = __int_as_float(r1.y); v[6] = __int_as_float(r1.z); v[7] = __int_as_float(r1.w);
}

// eight consecutive output samples t .. t + 7 (t a multiple of 8) of row b -> interleaved int16 PCM [clips, total, C]
__device__ __forceinline__ void pcm_store8(int16_t* pcm_out, int C, long b, long t, long total, const float (&v)[8]) {
  if (C == 1) {
    int4 w;
    int* wp = reinterpret_cast<int*>(&w);
#pragma unroll
    for (int i = 0; i < 4; ++i)
      wp[i] = (int)(uint16_t)pcm_quantise(v[2 * i]) | ((int)(uint16_t)pcm_quantise(v[2 * i + 1]) << 16);
    *reinterpret_cast<int4*>(pcm_out + (size_t)b * total + t) = w;
  } else {
    const long clip = b / C;
    const int ch = (int)(b - clip * C);
    int16_t* q = pcm_out + ((size_t)clip * total + t) * C + ch;
#pragma unroll
    for (int i = 0; i < 8; ++i) q[(size_t)i * C] = pcm_quantise(v[i]);
  }
}

}  // namespace pqmf
