// Direct-form PQMF kernels: bit-faithful to the registered bank `hk` for ANY n_band / L / T.
//
// These are the exactness reference inside the library and the path for everything the
// fold + tensor-core kernels (fast16.cuh) do not cover: n_band != 16, non power-of-two
// n_band in classic mode (reference pqmf.py:220-224 allows it), ragged T, PQMF_FLAG_EXACT.
//
//   analysis : y[b,k,n]  = sigma(k, n+par) * sum_j hk[k,j] * X[b, n*M + j - off]
//   synthesis: out[b,tau] = M * sum_k sum_n sigma(k, n+par) S[b,k,n] * hk[k, tau - n*M + off2]
//
// (closed forms of reference pqmf.py:115-130/160-177 and :133-157/180-199, SURVEY.md A.1.)
// X / S are the block optionally preceded by caller-owned history (streaming mode).  The POOL instantiations serve stream pools
// (stream_pool.cuh): row b is the next block of stream ids[b], whose history, next history and frame parity come from the pool and the
// stream's phase word; a row whose id is outside [0, P) gives zeros and touches no state.
//
// Both kernels are register-tiled correlations on a polyphase shared-memory layout:
// lanes walk consecutive frames (conflict-free LDS, coalesced sub-band rows), each thread owns
// 4 bands (analysis) or 4 output phases (synthesis) x RF frames, and the bank slice is read as
// one LDS.128 per tap.  They are CUDA-core kernels on purpose: 2*L flop/sample is far off the
// HBM roofline, and no tensor-core formulation of the direct form meets the 1e-5 budget within
// it (DESIGN.md section 4).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "pcm.cuh"
#include "stream_pool.cuh"

namespace pqmf {

constexpr int kDirectThreads = 256;


__host__ __device__ inline long floor_div(long a, long b) {
  long q = a / b;
  return (a % b != 0 && ((a < 0) != (b < 0))) ? q - 1 : q;
}

// ---------------------------------------------------------------------------------------------
// analysis
// ---------------------------------------------------------------------------------------------
struct AnalysisDirectParams {
  const float* x;     // [B, T]
  const float* hist;  // [B, L] or nullptr (zeros)
  float* y;           // [B, M, n_frames]
  const float* hk;    // [M, L]
  long T, n_frames;
  int M, L;
  int off;       // L/2 offline, L streaming
  int parity;    // global index of frame 0, & 1
  int nosign;    // 1: skip the sign mask (free-function API: polyphase_forward / classic_forward)
  int JC;        // taps per chunk, multiple of M
  int QC;        // JC / M
  int xstride;   // row stride (floats) of the polyphase x tile, odd
  int m_shift;   // log2(M) when M is a power of two, else -1
  PcmIn in;      // in.pcm != nullptr: the rows come from interleaved int16 PCM instead of x
  float* hist_out;  // streaming: the last L samples of (hist ++ x) per row (must not alias hist); the CTA of a row's last frame tile writes them
};
// POOL: hist and hist_out are both the pool [2, P, L]
struct AnalysisDirectPoolParams : AnalysisDirectParams {
  StreamPoolIndex pool;
};

template <int BG, int RF, bool POOL>
__global__ void __launch_bounds__(kDirectThreads) analysis_direct_kernel(std::conditional_t<POOL, AnalysisDirectPoolParams, AnalysisDirectParams> p) {
  constexpr int FL = kDirectThreads / BG;  // frame lanes
  constexpr int FT = FL * RF;              // frames per CTA
  constexpr int NB = 4 * BG;               // bands per CTA
  extern __shared__ __align__(16) float smem[];
  float* hsT = smem;                        // [JC][NB]
  float* xs = smem + (size_t)p.JC * NB;     // [M][xstride]

  const int tid = threadIdx.x;
  const int tf = tid % FL;
  const int bg = tid / FL;
  const long n0 = (long)blockIdx.x * FT;
  const int kb = blockIdx.y * NB;
  const int b = blockIdx.z;
  const int M = p.M, L = p.L;
  const float* xrow = p.x + (size_t)b * p.T;
  const float* hrow = p.hist ? p.hist + (size_t)b * L : nullptr;
  float* hout = nullptr;  // POOL: the stream's next history row
  int parity = 0;         // POOL: the stream's frame parity
  if constexpr (POOL) {
    size_t cur, next;
    if (!pool_row(p.pool, b, (size_t)L, cur, next, parity)) {  // dead row: zero sub-bands
      float* yb = p.y + (size_t)b * M * p.n_frames;
      for (int e = tid; e < FT * NB; e += kDirectThreads) {
        const long n = n0 + e % FT;
        const int k = kb + e / FT;
        if (n < p.n_frames && k < M) yb[(size_t)k * p.n_frames + n] = 0.f;
      }
      return;
    }
    hrow = p.hist + cur;
    hout = p.hist_out + next;
  }

  float acc[RF][4];
#pragma unroll
  for (int r = 0; r < RF; ++r)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[r][c] = 0.f;

  for (int j0 = 0; j0 < L; j0 += p.JC) {
    const int jc = min(p.JC, L - j0);
    __syncthreads();
    // bank slice, transposed to [tap][band] so one LDS.128 yields 4 bands of one tap
    for (int e = tid; e < p.JC * NB; e += kDirectThreads) {
      const int kk = e / p.JC, jj = e - kk * p.JC;  // coalesced along taps
      const int k = kb + kk;
      hsT[jj * NB + kk] = (k < M && jj < jc) ? __ldg(p.hk + (size_t)k * L + j0 + jj) : 0.f;
    }
    // x window in polyphase layout xs[u % M][u / M], u = local sample index
    const long base = n0 * M + j0 - p.off;
    const int U = (FT - 1) * M + p.JC;
    for (int u = tid; u < U; u += kDirectThreads) {
      const long s = base + u;
      float v = 0.f;
      if (s >= 0) {
        if (s < p.T) v = p.in.pcm ? pcm_sample(p.in, b, s, p.T) : __ldg(xrow + s);
      } else if (hrow != nullptr && s >= -(long)L) {
        v = __ldg(hrow + L + s);
      }
      int ph, i;
      if (p.m_shift >= 0) {
        ph = u & (M - 1);
        i = u >> p.m_shift;
      } else {
        i = u / M;
        ph = u - i * M;
      }
      xs[ph * p.xstride + i] = v;
    }
    __syncthreads();
    const float4* h4 = reinterpret_cast<const float4*>(hsT) + bg;
    for (int qq = 0; qq < p.QC; ++qq) {
      const float* xq = xs + tf + qq;
      const float4* hq = h4 + (size_t)qq * M * BG;
#pragma unroll 4
      for (int pp = 0; pp < M; ++pp) {
        const float4 hv = hq[pp * BG];
        const float* xp = xq + pp * p.xstride;
#pragma unroll
        for (int r = 0; r < RF; ++r) {
          const float xv = xp[r * FL];
          acc[r][0] = fmaf(hv.x, xv, acc[r][0]);
          acc[r][1] = fmaf(hv.y, xv, acc[r][1]);
          acc[r][2] = fmaf(hv.z, xv, acc[r][2]);
          acc[r][3] = fmaf(hv.w, xv, acc[r][3]);
        }
      }
    }
  }
  if (p.hist_out != nullptr && blockIdx.x == gridDim.x - 1 && blockIdx.y == 0) {  // streaming: roll this row's history (no extra launch)
    for (int i = tid; i < L; i += kDirectThreads) {
      const long src = (long)i + p.T - L;  // position in the block; negative: still inside the old history
      const float v = src >= 0 ? __ldg(xrow + src) : (hrow != nullptr ? __ldg(hrow + i + p.T) : 0.f);
      if constexpr (POOL) hout[i] = v;
      else p.hist_out[(size_t)b * L + i] = v;
    }
  }
  float* yb = p.y + (size_t)b * M * p.n_frames;
#pragma unroll
  for (int r = 0; r < RF; ++r) {
    const long n = n0 + tf + r * FL;
    if (n >= p.n_frames) continue;
    const bool even = !p.nosign && ((n + (POOL ? parity : p.parity)) & 1) == 0;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int k = kb + bg * 4 + c;
      if (k < M) {
        const float v = acc[r][c];
        yb[(size_t)k * p.n_frames + n] = (even && (k & 1)) ? -v : v;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// synthesis
// ---------------------------------------------------------------------------------------------
constexpr int kMaxBandTable = 64;

// ---- per-band hand-off of the pitch-shifter pipeline (SURVEY 8f-3; reference PitchShifterPvoc/1-PitchShifterWrapper.py:243-295).
// The n_band sub-bands arrive as SEPARATE tensors of different lengths (each band went through its own pitch shifter); the reference
// cross-fades the first Lx samples of every band with the tail kept from the previous block (:259-276), centre-crops or zero-pads
// every band to the frame count of the analysis (:279-289), concatenates them (:295) and only then calls inverse.  Here the synthesis
// kernel reads the bands through this table and applies cross-fade and crop/pad on the fly: no intermediate tensors. ----
struct BandTable {
  const float* band[kMaxBandTable];  // band k: [B, len[k]] row-contiguous
  int len[kMaxBandTable];
  int start[kMaxBandTable];          // frame f of the synthesis input is sample f + start[k] of band k (negative: left zero padding)
  const float* prev_tail;            // [M, Lx] or nullptr (no cross-fade)
  const float* fade_out;             // [Lx]
  const float* fade_in;              // [Lx]
  int Lx;
  int enabled;
};
// sub-band frame n of band k, row b, after cross-fade and crop/pad
__device__ __forceinline__ float band_value(const BandTable& t, int k, long b, long n) {
  const long u = n + t.start[k];
  if (u < 0 || u >= t.len[k]) return 0.f;
  float v = __ldg(t.band[k] + (size_t)b * t.len[k] + u);
  if (t.prev_tail != nullptr && u < t.Lx && t.len[k] >= t.Lx)
    v = __fadd_rn(__fmul_rn(__ldg(t.prev_tail + (size_t)k * t.Lx + u), __ldg(t.fade_out + u)), __fmul_rn(v, __ldg(t.fade_in + u)));  // torch: mul, mul, add
  return v;
}
// the tail kept for the next block: the last Lx samples of every band AFTER the cross-fade wrote its prefix (the reference reads the
// suffix through a view, so for len < 2 Lx it sees blended values); bands shorter than Lx leave their tail unchanged
__global__ void band_tail_kernel(BandTable t, int M, float* __restrict__ tail_out) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= M * t.Lx) return;
  const int k = idx / t.Lx, j = idx - k * t.Lx;
  float v = __ldg(t.prev_tail + idx);
  if (t.len[k] >= t.Lx) {
    const long u = (long)t.len[k] - t.Lx + j;
    v = __ldg(t.band[k] + u);
    if (u < t.Lx) v = __fadd_rn(__fmul_rn(__ldg(t.prev_tail + (size_t)k * t.Lx + u), __ldg(t.fade_out + u)), __fmul_rn(v, __ldg(t.fade_in + u)));
  }
  tail_out[idx] = v;
}

struct SynthesisDirectParams {
  const float* s;     // [B, M, F]
  const float* hist;  // [B, M, K] or nullptr
  float* out;         // [B, M*F]
  const float* hk;    // [M, L]
  long F;
  int M, L, K;        // K = frames of history (L / M), only used with hist
  int off2;           // L/2 - delay*M offline, -M streaming
  int parity;
  int nosign;
  int dlo, ND;        // tap-frame range d in [dlo, dlo + ND)
  int hstride;        // floats per band row of the padded bank slice (ND*M + 16)
  int sstride;        // floats per band row of the sub-band tile
  int16_t* pcm_out;   // != nullptr: write interleaved int16 PCM [clips, M F, C] (row = clip * C + channel) instead of out
  int C;
  BandTable bands;    // bands.enabled: the sub-bands come from n_band separate tensors (s unused)
  float* hist_out;    // streaming: the last K frames of (hist ++ s) per band row (must not alias hist), written by the row's last frame tile
};
// POOL: hist and hist_out are both the pool [2, P, M, K]
struct SynthesisDirectPoolParams : SynthesisDirectParams {
  StreamPoolIndex pool;
};

constexpr int kSynthBandsPerChunk = 4;
template <int PG, int RF, bool VEC, bool POOL>
__global__ void __launch_bounds__(kDirectThreads)
    synthesis_direct_kernel(std::conditional_t<POOL, SynthesisDirectPoolParams, SynthesisDirectParams> p) {
  constexpr int FL = kDirectThreads / PG;
  constexpr int FT = FL * RF;
  constexpr int NP = 4 * PG;  // output phases per CTA
  constexpr int KB = kSynthBandsPerChunk;
  extern __shared__ __align__(16) float smem[];
  float* hs = smem;                          // [KB][hstride]   hs[kk][(d-dlo)*M + phase]
  float* ss = smem + (size_t)KB * p.hstride;  // [KB][sstride]   ss[kk][n - nlo]

  const int tid = threadIdx.x;
  const int tf = tid % FL;
  const int pg = tid / FL;
  const long f0 = (long)blockIdx.x * FT;
  const int p0 = blockIdx.y * NP + pg * 4;
  const int b = blockIdx.z;
  const int M = p.M, L = p.L;
  const int dhi = p.dlo + p.ND - 1;
  const long nlo = f0 - dhi;
  const int NS = FT + p.ND - 1;
  const int jlo = p.dlo * M + p.off2;  // tap index of (d = dlo, phase 0)
  const float* sb = p.s + (size_t)b * M * p.F;
  const float* hb = p.hist ? p.hist + (size_t)b * M * p.K : nullptr;
  float* hout = nullptr;  // POOL: the stream's next history row
  int parity = 0;         // POOL: the stream's frame parity
  if constexpr (POOL) {
    size_t cur, next;
    if (!pool_row(p.pool, b, (size_t)M * p.K, cur, next, parity)) {  // dead row: zero output
      float* ob = p.out + (size_t)b * M * p.F;
      for (int e = tid; e < FT * NP; e += kDirectThreads) {
        const long f = f0 + e % FT;
        const int ph = blockIdx.y * NP + e / FT;
        if (f < p.F && ph < M) ob[f * M + ph] = 0.f;
      }
      return;
    }
    hb = p.hist + cur;
    hout = p.hist_out + next;
  }

  float acc[RF][4];
#pragma unroll
  for (int r = 0; r < RF; ++r)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[r][c] = 0.f;

  for (int k0 = 0; k0 < M; k0 += KB) {
    __syncthreads();
    const int HW = p.ND * M;
    for (int e = tid; e < KB * p.hstride; e += kDirectThreads) {
      const int kk = e / p.hstride, jj = e - kk * p.hstride;
      const int k = k0 + kk, j = jlo + jj;
      hs[e] = (k < M && jj < HW && j >= 0 && j < L) ? __ldg(p.hk + (size_t)k * L + j) : 0.f;
    }
    for (int e = tid; e < KB * NS; e += kDirectThreads) {
      const int kk = e / NS, i = e - kk * NS;
      const int k = k0 + kk;
      const long n = nlo + i;
      float v = 0.f;
      if (k < M) {
        if (n >= 0) {
          if (n < p.F) v = p.bands.enabled ? band_value(p.bands, k, b, n) : __ldg(sb + (size_t)k * p.F + n);
        } else if (hb != nullptr && n >= -(long)p.K) {
          v = __ldg(hb + (size_t)k * p.K + p.K + n);
        }
        if (!p.nosign && (k & 1) && (((n + (POOL ? parity : p.parity)) & 1) == 0)) v = -v;
      }
      ss[kk * p.sstride + i] = v;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < KB; ++kk) {
      const float* hrow = hs + kk * p.hstride + pg * 4 + blockIdx.y * NP;
      const float* srow = ss + kk * p.sstride + tf + dhi - p.dlo;  // index of d = dlo
#pragma unroll 4
      for (int dd = 0; dd < p.ND; ++dd) {
        float4 hv;
        if (VEC) {
          hv = *reinterpret_cast<const float4*>(hrow + dd * M);
        } else {
          hv.x = hrow[dd * M];
          hv.y = hrow[dd * M + 1];
          hv.z = hrow[dd * M + 2];
          hv.w = hrow[dd * M + 3];
        }
#pragma unroll
        for (int r = 0; r < RF; ++r) {
          const float sv = srow[r * FL - dd];
          acc[r][0] = fmaf(hv.x, sv, acc[r][0]);
          acc[r][1] = fmaf(hv.y, sv, acc[r][1]);
          acc[r][2] = fmaf(hv.z, sv, acc[r][2]);
          acc[r][3] = fmaf(hv.w, sv, acc[r][3]);
        }
      }
    }
  }
  if (p.hist_out != nullptr && blockIdx.x == gridDim.x - 1 && blockIdx.y == 0) {  // streaming: roll the sub-band history of this row
    for (int e = tid; e < M * p.K; e += kDirectThreads) {
      const int k = e / p.K, i = e - k * p.K;
      const long src = (long)i + p.F - p.K;
      const float v = src >= 0 ? __ldg(sb + (size_t)k * p.F + src) : (hb != nullptr ? __ldg(hb + (size_t)k * p.K + i + p.F) : 0.f);
      if constexpr (POOL) hout[(size_t)k * p.K + i] = v;
      else p.hist_out[((size_t)b * M + k) * p.K + i] = v;
    }
  }
  const float gain = (float)M;
  float* ob = p.out + (size_t)b * M * p.F;
#pragma unroll
  for (int r = 0; r < RF; ++r) {
    const long f = f0 + tf + r * FL;
    if (f >= p.F) continue;
    if (p.pcm_out != nullptr) {
      const long clip = b / p.C;
      const int ch = b - (int)(clip * p.C);
      int16_t* q = p.pcm_out + ((size_t)clip * M * p.F + f * M + p0) * p.C + ch;
#pragma unroll
      for (int c = 0; c < 4; ++c)
        if (p0 + c < M) q[(size_t)c * p.C] = pcm_quantise(acc[r][c] * gain);
      continue;
    }
    float* o = ob + f * M + p0;
    if (VEC && p0 + 3 < M) {
      *reinterpret_cast<float4*>(o) = make_float4(acc[r][0] * gain, acc[r][1] * gain, acc[r][2] * gain, acc[r][3] * gain);
    } else {
#pragma unroll
      for (int c = 0; c < 4; ++c)
        if (p0 + c < M) o[c] = acc[r][c] * gain;
    }
  }
}

}  // namespace pqmf
