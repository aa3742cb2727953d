// pqmf_b200 C ABI (include/pqmf_b200.h): argument checking, kernel selection, launches.
// No torch types, no allocation on the device-pointer entry points, no synchronisation.
#include "../../include/pqmf_b200.h"

#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <thread>
#include <type_traits>
#include <vector>

#include "direct_form.cuh"
#include "fast16.cuh"
#include "fast16_synth.cuh"
#include "hankel16.cuh"
#include "hankel4.cuh"
#include "hankel4_stream.cuh"

namespace {

std::atomic<unsigned long long> g_launches{0};

inline int log2_exact(int v) {
  if (v <= 0 || (v & (v - 1))) return -1;
  int s = 0;
  while ((1 << s) < v) ++s;
  return s;
}

inline int cuda_status() {
  cudaError_t e = cudaGetLastError();
  return (int)e;
}

template <typename K>
int ensure_smem(K kernel, size_t bytes) {
  if (bytes <= 48 * 1024) return 0;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  return (int)e;
}

// stream pools (stream_pool.cuh): the rows of a call are streams ids[0 .. n) of a pool of P
using PoolRows = pqmf::StreamPoolIndex;

// ------------------------------------------------------------------ direct-form launches
// Params: AnalysisDirectParams, or AnalysisDirectPoolParams for the POOL instantiations
template <int BG, int RF, typename Params>
int launch_analysis_direct(Params p, int B, cudaStream_t st) {
  constexpr bool POOL = std::is_same_v<Params, pqmf::AnalysisDirectPoolParams>;
  constexpr int FL = pqmf::kDirectThreads / BG, FT = FL * RF, NB = 4 * BG;
  p.xstride = (FT + p.QC - 1) | 1;
  const size_t smem = ((size_t)p.JC * NB + (size_t)p.M * p.xstride) * sizeof(float);
  if (smem > 200 * 1024) return PQMF_ERR_UNSUPPORTED;
  auto kern = pqmf::analysis_direct_kernel<BG, RF, POOL>;
  if (int e = ensure_smem(kern, smem)) return e;
  dim3 grid((unsigned)((p.n_frames + FT - 1) / FT), (unsigned)((p.M + NB - 1) / NB), (unsigned)B);
  kern<<<grid, pqmf::kDirectThreads, smem, st>>>(p);
  ++g_launches;
  return cuda_status();
}

int analysis_direct(const float* x, const float* hist, float* y, const float* hk, int B, long T, long n_frames, int M, int L,
                    int off, int parity, int nosign, cudaStream_t st, pqmf::PcmIn pcm = pqmf::PcmIn{nullptr, 1, 0}, float* hist_out = nullptr,
                    const PoolRows* pool = nullptr) {
  if (n_frames == 0 || B == 0) return PQMF_OK;
  pqmf::AnalysisDirectParams p{};
  p.x = x; p.hist = hist; p.y = y; p.hk = hk; p.in = pcm; p.hist_out = hist_out;
  p.T = T; p.n_frames = n_frames; p.M = M; p.L = L; p.off = off; p.parity = parity & 1; p.nosign = nosign;
  p.m_shift = log2_exact(M);
  int jc = (512 / M) * M;
  if (jc < M) jc = M;
  const int lceil = ((L + M - 1) / M) * M;
  if (jc > lceil) jc = lceil;
  p.JC = jc; p.QC = jc / M;
  if (B > 65535) return PQMF_ERR_UNSUPPORTED;
  if (pool) {
    const pqmf::AnalysisDirectPoolParams q{p, *pool};
    if (M <= 4) return launch_analysis_direct<1, 4>(q, B, st);
    if (M <= 8) return launch_analysis_direct<2, 4>(q, B, st);
    if (M <= 32) return launch_analysis_direct<4, 4>(q, B, st);
    if (M <= 64) return launch_analysis_direct<4, 2>(q, B, st);
    return launch_analysis_direct<4, 1>(q, B, st);
  }
  if (M <= 4) return launch_analysis_direct<1, 4>(p, B, st);
  if (M <= 8) return launch_analysis_direct<2, 4>(p, B, st);
  if (M <= 32) return launch_analysis_direct<4, 4>(p, B, st);
  if (M <= 64) return launch_analysis_direct<4, 2>(p, B, st);
  return launch_analysis_direct<4, 1>(p, B, st);
}

// Params: SynthesisDirectParams, or SynthesisDirectPoolParams for the POOL instantiations
template <int PG, int RF, bool VEC, typename Params>
int launch_synthesis_direct(Params p, int B, cudaStream_t st) {
  constexpr bool POOL = std::is_same_v<Params, pqmf::SynthesisDirectPoolParams>;
  constexpr int FL = pqmf::kDirectThreads / PG, FT = FL * RF, NP = 4 * PG;
  p.hstride = p.ND * p.M + 16;
  p.sstride = (FT + p.ND - 1) | 1;
  const size_t smem = (size_t)pqmf::kSynthBandsPerChunk * ((size_t)p.hstride + p.sstride) * sizeof(float);
  if (smem > 200 * 1024) return PQMF_ERR_UNSUPPORTED;
  auto kern = pqmf::synthesis_direct_kernel<PG, RF, VEC, POOL>;
  if (int e = ensure_smem(kern, smem)) return e;
  dim3 grid((unsigned)((p.F + FT - 1) / FT), (unsigned)((p.M + NP - 1) / NP), (unsigned)B);
  kern<<<grid, pqmf::kDirectThreads, smem, st>>>(p);
  ++g_launches;
  return cuda_status();
}

int synthesis_direct(const float* s, const float* hist, float* out, const float* hk, int B, long F, int M, int L, int off2,
                     int parity, int nosign, cudaStream_t st, int16_t* pcm_out = nullptr, int C = 1, const pqmf::BandTable* bands = nullptr,
                     float* hist_out = nullptr, const PoolRows* pool = nullptr) {
  if (F == 0 || B == 0) return PQMF_OK;
  pqmf::SynthesisDirectParams p{};
  p.s = s; p.hist = hist; p.out = out; p.hk = hk; p.pcm_out = pcm_out; p.C = C; p.hist_out = hist_out;
  if (bands) p.bands = *bands;
  p.F = F; p.M = M; p.L = L; p.K = L / M; p.off2 = off2; p.parity = parity & 1; p.nosign = nosign;
  p.dlo = (int)pqmf::floor_div(-(long)off2, M);
  const int dhi = (int)pqmf::floor_div((long)L - 1 - off2, M);
  p.ND = dhi - p.dlo + 1;
  if (B > 65535) return PQMF_ERR_UNSUPPORTED;
  const bool vec = (M % 4) == 0;
  if (pool) {
    const pqmf::SynthesisDirectPoolParams q{p, *pool};
    if (!vec) return launch_synthesis_direct<4, 4, false>(q, B, st);
    if (M <= 4) return launch_synthesis_direct<1, 4, true>(q, B, st);
    if (M <= 8) return launch_synthesis_direct<2, 4, true>(q, B, st);
    return launch_synthesis_direct<4, 4, true>(q, B, st);
  }
  if (!vec) return launch_synthesis_direct<4, 4, false>(p, B, st);
  if (M <= 4) return launch_synthesis_direct<1, 4, true>(p, B, st);
  if (M <= 8) return launch_synthesis_direct<2, 4, true>(p, B, st);
  return launch_synthesis_direct<4, 4, true>(p, B, st);
}

bool bad_dims(int B, long n, int M, int L) { return B < 0 || n < 0 || M < 2 || L < M || L > (1 << 16); }

// per-device staging workspace of the host-buffer entry points (pqmf_roundtrip_host_*).  One mutex PER DEVICE: calls for different
// devices run concurrently (pqmf_roundtrip_host_multi_f32 drives every GPU of the box from one process, one host thread each).
constexpr int kHostSlots = 8, kMaxDevices = 16;  // upper bound; the calls cycle through n_slots of them (roundtrip_host)
struct HostWorkspace {
  std::mutex mutex;
  cudaStream_t st[kHostSlots] = {};    // copy streams
  cudaStream_t kst[kHostSlots] = {};   // kernel streams
  cudaEvent_t up[kHostSlots] = {}, kdone[kHostSlots] = {}, down[kHostSlots] = {};  // H2D landed / kernels finished / D2H finished, per slot
  cudaEvent_t bank_up = nullptr;       // this call's bank and tables have landed
  void* d_x[kHostSlots] = {};   // input chunk (fp32 rows or int16 WAV frames)
  float* d_y[kHostSlots] = {};  // sub-bands of the chunk
  void* d_o[kHostSlots] = {};   // output chunk
  float* d_bank = nullptr;
  size_t chunk_elems = 0, bank_elems = 0;
  bool streams_ready = false;
};
HostWorkspace g_host_ws[kMaxDevices];

// Worst-case error the trimmed correction steps of the Hankel kernels may add, per unit of max|input| (hankel4_pick_trim).  Derived
// from north_star's 1e-5 max-abs tolerance against the reference's fp32 output (tools/trim_budget.py prints the table behind it):
// analysis 6e-6 -> 5 K-steps per side at the default bank (bound 5.7e-6; measured on audio-scale noise 1.2e-7 rms, 6.4e-7 max, on
// the adversarial sign-matched signal 1.6e-6); synthesis 1.5e-5 for ALL n_band sub-bands at |s| = 1 with adversarial signs, i.e.
// 9.8e-6 at the |s| <= 0.65 that sub-bands of audio reach (flute.wav: 0.65) -> 3 K-steps per side (bound 1.44e-5; measured on the
// reference's sub-bands 6.3e-8 rms, 3.7e-7 max; all bands at full scale with random signs 2.7e-6).  PQMF_FLAG_EXACT keeps every term.
constexpr double kTrimBudgetAnalysis = 6e-6, kTrimBudgetSynthesis = 1.5e-5;

constexpr long kFoldTableFloats = 512 + 2 * 16 * 32;  // [ g | c1 | c2 ] of the fold + modulation path
constexpr long kH16ImageFloats = 512L * 16;            // one hankel16 bank image (fp16 [KT/8][32][8]), sized for KT = 512
constexpr long kH4TableOffset = kFoldTableFloats + 2 * kH16ImageFloats;
constexpr long kH4ImageFloats = 35L * 4096 / 4;        // one hankel4 bank image (fp16 [2 KS][128][8]), sized for KS = 35
constexpr long kH4PairOffset = kH4TableOffset + 2 * kH4ImageFloats;
constexpr long kH4PairImageFloats = 2L * 35 * 3072 / 4;  // per-rank images of the CTA-pair kernels (fp16 [2][2 KS][96][8])

// ---- offline default for n_band 8 / 16 / 32 / 64: the 64-samples-per-row Hankel GEMM (hankel4.cuh) when there are enough tiles ----
// prototype lengths: L = 32 M at attenuation ~100, 16 M / 64 M for shorter / longer designs
bool h4_family(int M, int L) { return (M == 4 || M == 8 || M == 16 || M == 32 || M == 64) && (L == 16 * M || L == 32 * M || L == 64 * M); }
int h4_ks(int M, int kt) { return (kt + 64 - M + 15) / 16; }
// one CTA-pair image = [2 ranks][2 ks][96 rows][8] fp16 = 1536 ks floats.  Region sizes are fixed by (M, L) alone: a bank that
// fits one SM uses [analysis | synthesis], sized for kt = L; a longer one is SPLIT into two tap ranges that run as two launches
// (the second accumulates): [analysis lo | analysis hi | synthesis lo | synthesis hi], each sized for kt = L / 2.
// n_band 4: a frame is 8 bytes, but operand windows start on 16-byte boundaries, so the synthesis alignment pad must be an even
// number of frames; the tables therefore hold TWO synthesis images (largest lag ehi and ehi + 1) and the launch picks the one
// that makes (o - ehi) even.  Image regions are sized for that one extra frame of lag.
long h4_pair_floats(int M, int L) { return 1536L * h4_ks(M, L + (M < 8 ? M : 0)); }
long h4_half_floats(int M, int L) { return 1536L * h4_ks(M, L / 2); }
long h4_pair_offset(int M, int L) { return pqmf::hankel16_supported(M, L) ? kH4PairOffset : 0; }  // those tables start with the fold / Hankel-16 parts
long h4_tables_floats(int M, int L) {
  const long whole = (M < 8 ? 3 : 2) * h4_pair_floats(M, L), split = 4 * h4_half_floats(M, L);
  return whole > split ? whole : split;
}
bool use_h4(int B, long F, int M, const float* hist) {
  return hist == nullptr && (long)B * (((long)F * M + pqmf::kH4TileSamples - 1) / pqmf::kH4TileSamples) >= 96;
}
// taps kept by the images in `tables` (PQMF_FLAG_TAPS from pqmf_build_tables_f32); kt == 0: the caller did not pass them.
// With PQMF_FLAG_H4_SPLIT the field holds half the span.
void h4_taps(unsigned flags, int& jlo, int& kt) {
  jlo = 32 * (int)((flags >> 8) & 0xF);
  kt = 32 * (int)((flags >> 12) & 0x1F);
}

template <int M>
int h4_analysis_m(pqmf::H4AnalysisParams p, const float* tables, int jlo, int kt, int B, int L, unsigned flags, cudaStream_t st, pqmf::H4Io io) {
  const int trim = (flags & PQMF_FLAG_EXACT) ? 0 : (int)PQMF_FLAG_H4_TRIM_A(flags);  // exact mode: every correction term
  if (flags & PQMF_FLAG_H4_SPLIT) {  // two tap ranges, two launches; only the outer edge of each range may skip the corrections
    for (int half = 0; half < 2; ++half) {
      p.g = pqmf::h4_shape(M, jlo + half * kt, kt, true, false);
      p.bank = reinterpret_cast<const uint16_t*>(tables + h4_pair_offset(M, L) + half * h4_half_floats(M, L));
      p.trim_lo = half ? 0 : trim;
      p.trim_hi = half ? trim : 0;
      p.accumulate = half;
      if (const int e = pqmf::h4_launch_analysis<M, true>(p, B, st, io)) {
        if (half) return e;
        (void)cudaGetLastError();  // nothing was launched: the caller falls back to the direct form, which must not see this error
        return PQMF_ERR_UNSUPPORTED;
      }
    }
    return 0;
  }
  p.trim_lo = p.trim_hi = trim;
  if (!(flags & PQMF_FLAG_NO_PAIR)) {
    p.g = pqmf::h4_shape(M, jlo, kt, true, false);
    p.bank = reinterpret_cast<const uint16_t*>(tables + h4_pair_offset(M, L));
    const int e = pqmf::h4_launch_analysis<M, true>(p, B, st, io);
    if (e == 0) return 0;
    (void)cudaGetLastError();  // a context that cannot co-schedule CTA pairs (e.g. an SM partition): same arithmetic, one CTA per SM
  }
  if constexpr (M != 16) {
    return PQMF_ERR_UNSUPPORTED;  // single-CTA images are only built for n_band 16 / L 512
  } else {
    if (!pqmf::hankel16_supported(M, L)) return PQMF_ERR_UNSUPPORTED;
    p.g = pqmf::h4_shape(M, jlo, kt, false, false);
    p.bank = reinterpret_cast<const uint16_t*>(tables + kH4TableOffset);
    return pqmf::h4_launch_analysis<M, false>(p, B, st, io);
  }
}
// x / y: float32 rows and sub-bands, or raw half bits when io is F16 / BF16 (x unused with PCM input)
int h4_analysis(const void* x, void* y, const float* tables, int B, long T, long F, int M, int L, unsigned flags, cudaStream_t st,
                pqmf::PcmIn pcm = pqmf::PcmIn{nullptr, 1, 0}, pqmf::H4Io io = pqmf::H4Io::F32) {
  int jlo, kt;
  h4_taps(flags, jlo, kt);
  if (kt == 0) return PQMF_ERR_UNSUPPORTED;
  pqmf::H4AnalysisParams p{};
  p.x = static_cast<const float*>(x); p.in = pcm; p.y = static_cast<float*>(y); p.T = T; p.F = F; p.off = L / 2; p.parity = 0; p.keep_in_l2 = 1;
  switch (M) {
    case 4: return h4_analysis_m<4>(p, tables, jlo, kt, B, L, flags, st, io);
    case 8: return h4_analysis_m<8>(p, tables, jlo, kt, B, L, flags, st, io);
    case 16: return h4_analysis_m<16>(p, tables, jlo, kt, B, L, flags, st, io);
    case 32: return h4_analysis_m<32>(p, tables, jlo, kt, B, L, flags, st, io);
    case 64: return h4_analysis_m<64>(p, tables, jlo, kt, B, L, flags, st, io);
    default: return PQMF_ERR_UNSUPPORTED;
  }
}

template <int M>
int h4_synthesis_m(pqmf::H4SynthesisParams p, const float* tables, int jlo, int kt, int B, int L, unsigned flags, cudaStream_t st, pqmf::H4Io io) {
  const int trim = (flags & PQMF_FLAG_EXACT) ? 0 : (int)PQMF_FLAG_H4_TRIM_S(flags);
  if ((flags & PQMF_FLAG_H4_SPLIT) && p.pcm_out != nullptr) return PQMF_ERR_UNSUPPORTED;  // the second launch accumulates: not in int16
  if (flags & PQMF_FLAG_H4_SPLIT) {
    for (int half = 0; half < 2; ++half) {
      p.g = pqmf::h4_shape(M, jlo + half * kt, kt, true, true);
      p.bank = reinterpret_cast<const uint16_t*>(tables + h4_pair_offset(M, L) + (2 + half) * h4_half_floats(M, L));
      // synthesis K-steps run from the largest lag (the END of the tap range) down: the outer edge of the low range is its last steps
      p.trim_lo = half ? trim : 0;
      p.trim_hi = half ? 0 : trim;
      p.accumulate = half;
      if (const int e = pqmf::h4_launch_synthesis<M, true>(p, B, st, io)) {
        if (half) return e;
        (void)cudaGetLastError();
        return PQMF_ERR_UNSUPPORTED;
      }
    }
    return 0;
  }
  p.trim_lo = p.trim_hi = trim;
  if (!(flags & PQMF_FLAG_NO_PAIR)) {
    // n_band 4: the image whose largest lag makes (o - ehi) even (see h4_pair_floats); its K-steps sit one frame later, so give
    // up one trimmed step to stay inside the error budget that was computed for the other image
    const int variant = (M < 8) ? ((p.o - ((jlo + kt) / M - 1)) & 1) : 0;
    if (variant) p.trim_lo = p.trim_hi = trim > 0 ? trim - 1 : 0;
    p.g = pqmf::h4_shape(M, jlo, kt + variant * M, true, true);
    p.bank = reinterpret_cast<const uint16_t*>(tables + h4_pair_offset(M, L) + (1 + variant) * h4_pair_floats(M, L));
    const int e = pqmf::h4_launch_synthesis<M, true>(p, B, st, io);
    if (e == 0) return 0;
    (void)cudaGetLastError();
  }
  if constexpr (M != 16) {
    return PQMF_ERR_UNSUPPORTED;
  } else {
    if (!pqmf::hankel16_supported(M, L)) return PQMF_ERR_UNSUPPORTED;
    p.g = pqmf::h4_shape(M, jlo, kt, false, true);
    p.bank = reinterpret_cast<const uint16_t*>(tables + kH4TableOffset + kH4ImageFloats);
    return pqmf::h4_launch_synthesis<M, false>(p, B, st, io);
  }
}
// s / out: float32 sub-bands and rows, or raw half bits when io is F16 / BF16 (out unused with PCM output)
int h4_synthesis(const void* s, void* out, const float* tables, int B, long F, int off2, int M, int L, unsigned flags, cudaStream_t st,
                 int16_t* pcm_out = nullptr, int C = 1, pqmf::H4Io io = pqmf::H4Io::F32) {
  int jlo, kt;
  h4_taps(flags, jlo, kt);
  if (kt == 0 || off2 % M != 0) return PQMF_ERR_UNSUPPORTED;
  pqmf::H4SynthesisParams p{};
  p.s = static_cast<const float*>(s); p.out = static_cast<float*>(out); p.pcm_out = pcm_out; p.C = C; p.F = F; p.o = off2 / M; p.parity = 0; p.reverse = 1;
  switch (M) {
    case 4: return h4_synthesis_m<4>(p, tables, jlo, kt, B, L, flags, st, io);
    case 8: return h4_synthesis_m<8>(p, tables, jlo, kt, B, L, flags, st, io);
    case 16: return h4_synthesis_m<16>(p, tables, jlo, kt, B, L, flags, st, io);
    case 32: return h4_synthesis_m<32>(p, tables, jlo, kt, B, L, flags, st, io);
    case 64: return h4_synthesis_m<64>(p, tables, jlo, kt, B, L, flags, st, io);
    default: return PQMF_ERR_UNSUPPORTED;
  }
}

// ---- streaming blocks on the Hankel-4 kernels (hankel4_stream.cuh): several streams per MMA tile.  ONE routing decision per direction
//      for every streaming entry -- lockstep and pool, fp32 and int16 PCM: the kernels serve a call exactly where h4_stream_family holds
//      and h4_*_stream_plan accepts its shape, flags and tile count, and its buffers meet the kernels' alignment (h4_*_stream_ok).
//      Everywhere else (short blocks, few streams, odd sizes) an fp32 call runs other kernels -- the fold kernels for lockstep n_band 16,
//      the direct form -- and a PCM call is refused with PQMF_ERR_UNSUPPORTED ----
bool use_fast(int M, int L, const float* tables, unsigned flags);
bool use_h4_family(int M, int L, const float* tables, unsigned flags);
bool h4_stream_family(int M, int L, const float* tables, unsigned flags) {
  if (use_fast(M, L, tables, flags)) return true;  // n_band 16 / L 512
  return !pqmf::hankel16_supported(M, L) && use_h4_family(M, L, tables, flags) && (M == 8 || M == 32);
}
// p: everything but the buffers and the parity
bool h4_analysis_stream_plan(int B, long T, int M, int L, const float* tables, unsigned flags, pqmf::H4AnalysisStreamParams& p) {
  if (!h4_stream_family(M, L, tables, flags)) return false;
  int jlo, kt;
  h4_taps(flags, jlo, kt);
  if (kt == 0 || (flags & (PQMF_FLAG_H4_SPLIT | PQMF_FLAG_NO_PAIR | PQMF_FLAG_FOLD))) return false;
  // the region of a stream starts with its history as WHOLE plane rows: where the taps need a fraction of a row (n_band 8: 224 samples)
  // the region carries the next multiple of 64 (the state holds L samples) and every window starts that much later (pad_bytes)
  const int hist = ((L - jlo + 63) / 64) * 64;
  if (hist > L || T % 256 != 0 || T < L || L % 8 != 0) return false;
  const pqmf::H4StreamGeom sg = pqmf::h4_stream_geom(T, hist);
  if (sg.pitch > pqmf::kH4Rows || sg.spt < 1 || (B + sg.spt - 1) / sg.spt < 96) return false;
  p.T = T; p.B = B; p.L = L;
  p.trim_lo = p.trim_hi = (flags & PQMF_FLAG_EXACT) ? 0 : (int)PQMF_FLAG_H4_TRIM_A(flags);
  p.pad_bytes = 2 * (hist - (L - jlo));
  p.g = pqmf::h4_shape(M, jlo, kt, true, false, p.pad_bytes);
  p.s = sg;
  p.bank = reinterpret_cast<const uint16_t*>(tables + h4_pair_offset(M, L));
  return pqmf::h4_shape_fits(p.g);
}
// 256-bit signal loads (a PCM block: 16-byte mono, 32-byte stereo loads), 128-bit sub-band stores and state accesses
bool h4_analysis_stream_ok(int B, long T, int M, int L, const float* tables, unsigned flags, const void* signal, const float* y, const float* state_in,
                           const float* state_out, pqmf::H4AnalysisStreamParams& p) {
  return h4_analysis_stream_plan(B, T, M, L, tables, flags, p) && ((uintptr_t)signal | (uintptr_t)state_in) % 32 == 0 &&
         ((uintptr_t)y | (uintptr_t)state_out) % 16 == 0;
}
bool h4_synthesis_stream_plan(int B, long F, int M, int L, const float* tables, unsigned flags, pqmf::H4SynthesisStreamParams& p) {
  if (!h4_stream_family(M, L, tables, flags)) return false;
  int jlo, kt;
  h4_taps(flags, jlo, kt);
  if (kt == 0 || (flags & (PQMF_FLAG_H4_SPLIT | PQMF_FLAG_NO_PAIR | PQMF_FLAG_FOLD))) return false;
  const int K = L / M, taps_frames = (jlo + kt) / M;  // = ehi + 1: with o = -1 the window of output frame f starts at sub-band frame f - taps_frames
  // history and block are whole plane rows (64 / M frames each) and whole frame quads: the region carries the history rounded up to
  // rows (the state holds K frames) and the windows start that many frames later (pad_bytes)
  const int hist_frames = ((taps_frames * M + 63) / 64) * 64 / M;
  if (hist_frames % 4 != 0 || hist_frames > K || (F * M) % 256 != 0 || F % 4 != 0 || F < K) return false;
  const pqmf::H4StreamGeom sg = pqmf::h4_stream_geom(F * M, hist_frames * M);
  if (sg.pitch > pqmf::kH4Rows || sg.spt < 1 || (B + sg.spt - 1) / sg.spt < 96) return false;
  p.F = F; p.B = B; p.K = K;
  p.trim_lo = p.trim_hi = (flags & PQMF_FLAG_EXACT) ? 0 : (int)PQMF_FLAG_H4_TRIM_S(flags);
  p.pad_bytes = 2 * M * (hist_frames - taps_frames);
  p.g = pqmf::h4_shape(M, jlo, kt, true, true, p.pad_bytes);
  p.sg = sg;
  p.bank = reinterpret_cast<const uint16_t*>(tables + h4_pair_offset(M, L) + h4_pair_floats(M, L));
  return pqmf::h4_shape_fits(p.g);
}
// 128-bit sub-band loads and state accesses; 256-bit fp32 output stores (PCM output: 128-bit int16 stores)
bool h4_synthesis_stream_ok(int B, long F, int M, int L, const float* tables, unsigned flags, const float* s, const void* out, bool pcm_out,
                            const float* state_in, const float* state_out, pqmf::H4SynthesisStreamParams& p) {
  return h4_synthesis_stream_plan(B, F, M, L, tables, flags, p) && ((uintptr_t)s | (uintptr_t)state_in | (uintptr_t)state_out) % 16 == 0 &&
         (uintptr_t)out % (pcm_out ? 16 : 32) == 0;
}
template <typename Params>
int h4_analysis_stream_launch(const Params& p, int M, cudaStream_t st) {
  switch (M) {
    case 8: return pqmf::h4_launch_analysis_stream<8>(p, st);
    case 16: return pqmf::h4_launch_analysis_stream<16>(p, st);
    case 32: return pqmf::h4_launch_analysis_stream<32>(p, st);
    default: return PQMF_ERR_UNSUPPORTED;
  }
}
template <typename Params>
int h4_synthesis_stream_launch(const Params& p, int M, cudaStream_t st) {
  switch (M) {
    case 8: return pqmf::h4_launch_synthesis_stream<8>(p, st);
    case 16: return pqmf::h4_launch_synthesis_stream<16>(p, st);
    case 32: return pqmf::h4_launch_synthesis_stream<32>(p, st);
    default: return PQMF_ERR_UNSUPPORTED;
  }
}
// pool != nullptr: the indexed (POOL) kernels, with state_in = state_out = the pool.  pcm != nullptr: the block is int16 WAV frames (x
// unused).  Returns 0, PQMF_ERR_UNSUPPORTED (refused: nothing launched) or the error of a launch that did not start (cleared).
int h4_analysis_stream(const float* x, float* y, const float* tables, const float* state_in, float* state_out, int B, long T, int M, int L,
                       int parity, unsigned flags, cudaStream_t st, const PoolRows* pool = nullptr, const pqmf::PcmIn* pcm = nullptr) {
  pqmf::H4AnalysisStreamParams p{};
  if (!h4_analysis_stream_ok(B, T, M, L, tables, flags, pcm ? static_cast<const void*>(pcm->pcm) : x, y, state_in, state_out, p))
    return PQMF_ERR_UNSUPPORTED;
  p.x = x; p.hist_in = state_in; p.hist_out = state_out; p.y = y; p.parity = parity & 1;
  int e;
  if (pcm && pool) e = h4_analysis_stream_launch(pqmf::H4AnalysisStreamPoolPcmParams{{p, *pool}, *pcm}, M, st);
  else if (pcm) e = h4_analysis_stream_launch(pqmf::H4AnalysisStreamPcmParams{p, *pcm}, M, st);
  else if (pool) e = h4_analysis_stream_launch(pqmf::H4AnalysisStreamPoolParams{p, *pool}, M, st);
  else e = h4_analysis_stream_launch(p, M, st);
  if (e != 0) (void)cudaGetLastError();
  return e;
}
// pcm_out != nullptr: mono int16 output rows (out unused)
int h4_synthesis_stream(const float* s, float* out, const float* tables, const float* state_in, float* state_out, int B, long F, int M, int L,
                        int parity, unsigned flags, cudaStream_t st, const PoolRows* pool = nullptr, int16_t* pcm_out = nullptr) {
  pqmf::H4SynthesisStreamParams p{};
  if (!h4_synthesis_stream_ok(B, F, M, L, tables, flags, s, pcm_out ? static_cast<const void*>(pcm_out) : out, pcm_out != nullptr, state_in,
                              state_out, p))
    return PQMF_ERR_UNSUPPORTED;
  p.s = s; p.state_in = state_in; p.state_out = state_out; p.out = out; p.parity = parity & 1;
  int e;
  if (pcm_out && pool) e = h4_synthesis_stream_launch(pqmf::H4SynthesisStreamPoolPcmParams{{p, *pool}, pcm_out}, M, st);
  else if (pcm_out) e = h4_synthesis_stream_launch(pqmf::H4SynthesisStreamPcmParams{p, pcm_out}, M, st);
  else if (pool) e = h4_synthesis_stream_launch(pqmf::H4SynthesisStreamPoolParams{p, *pool}, M, st);
  else e = h4_synthesis_stream_launch(p, M, st);
  if (e != 0) (void)cudaGetLastError();
  return e;
}

// n_band 16 fast path: fold + tensor-core modulation (fast16*.cuh), or -- with PQMF_FLAG_EXACT -- the direct form as an
// implicit-Hankel GEMM on the tensor cores (hankel16.cuh).  flags bits [8,12) = first active tap / 32, [12,17) = taps / 32.
int exact_tc_analysis(const float* x, const float* hist, float* y, float* hist_out, const float* tables, int B, long T, long F, int off,
                  int parity, unsigned flags, cudaStream_t st) {
  const bool trimmed = ((flags >> 8) & 0xF) == 2 && ((flags >> 12) & 0x1F) == 12;
  pqmf::H16AnalysisParams p{};
  p.x = x; p.hist = hist; p.y = y; p.hist_out = hist_out;
  p.bank = reinterpret_cast<const uint16_t*>(tables + kFoldTableFloats);
  p.T = T; p.F = F; p.off = off; p.parity = parity & 1;
  p.tiles_per_row = (F + pqmf::kH16Frames - 1) / pqmf::kH16Frames;
  p.n_tiles = p.tiles_per_row * B;
  if (hist != nullptr && ((uintptr_t)hist % 16 || (uintptr_t)hist_out % 16)) return PQMF_ERR_UNSUPPORTED;
  return trimmed ? pqmf::h16_launch_analysis<64, 384>(p, st) : pqmf::h16_launch_analysis<0, 512>(p, st);
}

int exact_tc_synthesis(const float* s, const float* hist, float* out, float* hist_out, const float* tables, int B, long F, int off2,
                   int parity, unsigned flags, cudaStream_t st) {
  const bool trimmed = ((flags >> 8) & 0xF) == 2 && ((flags >> 12) & 0x1F) == 12;
  const int kt = trimmed ? 384 : 512;
  if (off2 % 16 != 0) return PQMF_ERR_UNSUPPORTED;
  pqmf::H16SynthesisParams p{};
  p.s = s; p.hist = hist; p.out = out; p.hist_out = hist_out;
  p.bank = reinterpret_cast<const uint16_t*>(tables + kFoldTableFloats) + (size_t)kt * 32;
  p.F = F; p.o = off2 / 16; p.parity = parity & 1;
  p.tiles_per_row = (F + pqmf::kH16Frames - 1) / pqmf::kH16Frames;
  p.n_tiles = p.tiles_per_row * B;
  return trimmed ? pqmf::h16_launch_synthesis<64, 384>(p, st) : pqmf::h16_launch_synthesis<0, 512>(p, st);
}

// (offline calls try the Hankel-4 kernels before these: h4_route_analysis / h4_route_synthesis)
int fast_analysis(const float* x, const float* hist, float* y, float* hist_out, const float* tables, int B, long T, long F, int off,
                  int parity, unsigned flags, cudaStream_t st) {
  if (flags & (PQMF_FLAG_EXACT | PQMF_FLAG_NO_FOLD)) return exact_tc_analysis(x, hist, y, hist_out, tables, B, T, F, off, parity, flags, st);
  return pqmf::fast16_analysis(x, hist, y, hist_out, tables, B, T, F, off, parity, flags, st);
}

int fast_synthesis(const float* s, const float* hist, float* out, float* hist_out, const float* tables, int B, long F, int off2,
                   int parity, unsigned flags, cudaStream_t st) {
  if (flags & (PQMF_FLAG_EXACT | PQMF_FLAG_NO_FOLD)) return exact_tc_synthesis(s, hist, out, hist_out, tables, B, F, off2, parity, flags, st);
  return pqmf::fast16_synthesis(s, hist, out, hist_out, tables, B, F, off2, parity, flags, st);
}

bool use_fast(int M, int L, const float* tables, unsigned flags) {
  return tables != nullptr && !(flags & (PQMF_FLAG_NO_SIGN | PQMF_FLAG_FP32)) && pqmf::hankel16_supported(M, L);
}
// other band counts / prototype lengths: only the offline Hankel kernels exist (streaming, small batches and the sign-less free
// functions use the direct form); PQMF_FLAG_EXACT keeps them but runs every correction term
bool use_h4_family(int M, int L, const float* tables, unsigned flags) {
  return tables != nullptr && !(flags & (PQMF_FLAG_NO_SIGN | PQMF_FLAG_FOLD | PQMF_FLAG_FP32)) && h4_family(M, L);
}

// ---- which kernels an offline call runs: the offline Hankel-4 kernels exactly when these say so and the buffers are aligned for
//      them; everything else (n_band 16: the fold / Hankel-16 kernels; other band counts: the direct form) comes after.  The fp32 and
//      the half-precision entry points both decide here, so a half-precision call runs natively exactly where the fp32 call on its
//      widened input runs the same kernels with the same trims -- which is what makes the two bit-identical.
//      (n_band 16 / L 512: fast_analysis's shape checks, hankel16_analysis_ok, are implied.) ----
bool h4_route_analysis(int B, long T, long F, int M, int L, const float* tables, unsigned flags) {
  const bool shape = T > 0 && (T % M) == 0 && (T % 8) == 0 && F == T / M && use_h4(B, F, M, nullptr);
  if (use_fast(M, L, tables, flags)) return shape && !(flags & PQMF_FLAG_FOLD);
  return !pqmf::hankel16_supported(M, L) && use_h4_family(M, L, tables, flags) && shape;
}
bool h4_route_synthesis(int B, long F, int M, int L, const float* tables, unsigned flags) {
  const bool shape = F > 0 && (F & 3) == 0 && use_h4(B, F, M, nullptr);
  if (use_fast(M, L, tables, flags)) return shape && !(flags & PQMF_FLAG_FOLD);
  return !pqmf::hankel16_supported(M, L) && use_h4_family(M, L, tables, flags) && shape;
}
// fp32 buffers: 256-bit signal loads / stores, 128-bit sub-band loads / stores
bool h4_aligned_f32(const void* signal, const void* bands) { return ((uintptr_t)signal % 32) == 0 && ((uintptr_t)bands % 16) == 0; }
// half-precision buffers: 128-bit signal loads / stores; 64-bit sub-band loads, up to 128-bit sub-band stores
bool h4_aligned_half(const void* signal, const void* bands) { return (((uintptr_t)signal | (uintptr_t)bands) % 16) == 0; }
// the half-precision instantiations exist for the unsplit banks, as CTA pairs
bool half_analysis_native(const void* x, const void* y, int B, long T, long F, int M, int L, const float* tables, unsigned flags) {
  return h4_route_analysis(B, T, F, M, L, tables, flags) && !(flags & PQMF_FLAG_H4_SPLIT) && h4_aligned_half(x, y);
}
bool half_synthesis_native(const void* s, const void* out, int B, long F, int M, int L, const float* tables, unsigned flags) {
  return h4_route_synthesis(B, F, M, L, tables, flags) && !(flags & PQMF_FLAG_H4_SPLIT) && h4_aligned_half(out, s);
}
bool half_io_of(int dtype, pqmf::H4Io& io) {
  if (dtype == PQMF_DTYPE_F16) io = pqmf::H4Io::F16;
  else if (dtype == PQMF_DTYPE_BF16) io = pqmf::H4Io::BF16;
  else return false;
  return true;
}

// ---- chunk schedule of the host-buffer entry points (host arithmetic only; exported as pqmf_host_chunk_plan for the tests) ----
// Chunks of ~chunk_bytes of fp32 samples, whole clips, small chunks at both ends (1/4, 1/4, 1/2 of a chunk ...: nothing overlaps the
// first H2D copy and the last D2H copy), and never fewer clips than the 96 tiles of 8192 samples the Hankel kernels take (use_h4):
// a smaller chunk -- or a smaller remainder at the end -- would run other kernels, slower and with different rounding.
struct HostChunks {
  long clips_per_chunk, min_clips;
  long buffer_clips() const { return clips_per_chunk + min_clips - 1; }  // the largest chunk: a full one plus an undersized remainder
};
long host_chunk_bytes() {
  static const long v = [] {
    const char* e = getenv("PQMF_HOST_CHUNK_MIB");   // tuning knob; default 8 MiB of fp32 samples per chunk
    const long m = e ? atol(e) : 0;
    return (m > 0 && m <= 1024 ? m : 8L) << 20;
  }();
  return v;
}
HostChunks host_chunks(long B, long T, int C) {
  HostChunks h;
  const long tiles_per_clip = (long)C * ((T + pqmf::kH4TileSamples - 1) / pqmf::kH4TileSamples);
  h.min_clips = (96 + tiles_per_clip - 1) / tiles_per_clip;
  h.clips_per_chunk = host_chunk_bytes() / (T * C * (long)sizeof(float));
  if (h.clips_per_chunk < h.min_clips) h.clips_per_chunk = h.min_clips;
  if (h.clips_per_chunk > B) h.clips_per_chunk = B;
  return h;
}
long host_next_chunk(const HostChunks& h, long B, long r0) {  // clips in the chunk that starts at clip r0
  const long left = B - r0, done = r0, full = h.clips_per_chunk;
  const long ramp_in = done < full ? (done < 2 ? full / 4 : full / 2) : full;
  const long ramp_out = left <= full ? (left <= full / 2 ? full / 4 : full / 2) : full;
  long want = ramp_in < ramp_out ? ramp_in : ramp_out;
  if (want < h.min_clips) want = h.min_clips;
  long clips = left < want ? left : want;
  if (left - clips > 0 && left - clips < h.min_clips) clips = left;  // no undersized remainder: at most full + min_clips - 1 clips (buffer_clips)
  return clips;
}

// ---- host-buffer round trip, generic over the sample format (float rows, or int16 interleaved WAV frames with C channels) ----
// Row chunks of ~8 MiB of fp32 samples (2 Mi samples): the H2D copy of chunk i + 1, the two kernels of chunk i and the D2H copy of
// chunk i - 1 overlap (PCIe is full duplex); copies and kernels have streams of their own (see the copy-phase note in the loop below).
// The staging buffers live in a per-device workspace that is created on first use and only ever grows, so
// steady-state calls do no allocation.
template <typename Sample>
int roundtrip_host(const Sample* x_host, float* y_host, Sample* out_host, const float* hk_host, const float* tables_host, int B, long T, int C,
                   int M, int L, int delay_frames, unsigned flags, int device) {
  constexpr bool kPcm = sizeof(Sample) == 2;
  if (bad_dims(B, T, M, L) || !x_host || !out_host || !hk_host || (T % M) != 0) return PQMF_ERR_ARG;
  if (B == 0 || T == 0) return PQMF_OK;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev || device >= kMaxDevices) return PQMF_ERR_NO_DEVICE;
  cudaError_t e = cudaSetDevice(device);
  if (e != cudaSuccess) return (int)e;
  const long F = T / M;
  static const int n_slots = [] {
    const char* e = getenv("PQMF_HOST_SLOTS");       // tuning knob: chunks in flight (default 4)
    const int v = e ? atoi(e) : 0;
    return v >= 2 && v <= kHostSlots ? v : 4;
  }();
  const long clip_samples = T * C;                      // one clip = C rows of T samples
  const HostChunks plan = host_chunks(B, T, C);
  const long clips_per_chunk = plan.clips_per_chunk;
  const size_t chunk_elems = (size_t)(plan.buffer_clips() < B ? plan.buffer_clips() : B) * clip_samples;
  const long n_tab = tables_host ? pqmf_tables_numel(M, L) : 0;
  HostWorkspace& ws = g_host_ws[device];
  std::lock_guard<std::mutex> lock(ws.mutex);
  int rc = PQMF_OK;
  auto check = [&](cudaError_t err) { if (err != cudaSuccess && rc == PQMF_OK) rc = (int)err; return err == cudaSuccess; };
  if (!ws.streams_ready) {
    for (int i = 0; i < kHostSlots; ++i) {
      check(cudaStreamCreateWithFlags(&ws.st[i], cudaStreamNonBlocking));
      check(cudaStreamCreateWithFlags(&ws.kst[i], cudaStreamNonBlocking));
      check(cudaEventCreateWithFlags(&ws.up[i], cudaEventDisableTiming));
      check(cudaEventCreateWithFlags(&ws.kdone[i], cudaEventDisableTiming));
      check(cudaEventCreateWithFlags(&ws.down[i], cudaEventDisableTiming));
    }
    check(cudaEventCreateWithFlags(&ws.bank_up, cudaEventDisableTiming));
    ws.streams_ready = (rc == PQMF_OK);
  }
  if (rc == PQMF_OK && ws.chunk_elems < chunk_elems) {   // buffers are sized for fp32 samples: int16 chunks fit too
    for (int i = 0; i < kHostSlots; ++i) {
      if (ws.d_x[i]) cudaFree(ws.d_x[i]);
      if (ws.d_y[i]) cudaFree(ws.d_y[i]);
      if (ws.d_o[i]) cudaFree(ws.d_o[i]);
      ws.d_x[i] = ws.d_o[i] = nullptr;
      ws.d_y[i] = nullptr;
      if (i >= n_slots) continue;
      check(cudaMalloc(&ws.d_x[i], chunk_elems * sizeof(float)));
      check(cudaMalloc(&ws.d_y[i], chunk_elems * sizeof(float)));
      check(cudaMalloc(&ws.d_o[i], chunk_elems * sizeof(float)));
    }
    ws.chunk_elems = (rc == PQMF_OK) ? chunk_elems : 0;
  }
  const size_t bank_elems = (size_t)M * L;
  if (rc == PQMF_OK && ws.bank_elems < bank_elems + (size_t)n_tab) {
    if (ws.d_bank) cudaFree(ws.d_bank);
    ws.d_bank = nullptr;
    check(cudaMalloc(&ws.d_bank, (bank_elems + (size_t)n_tab) * sizeof(float)));
    ws.bank_elems = (rc == PQMF_OK) ? bank_elems + (size_t)n_tab : 0;
  }
  if (rc != PQMF_OK) return rc;
  float* d_hk = ws.d_bank;
  float* d_tab = n_tab ? ws.d_bank + bank_elems : nullptr;
  // the bank is tiny (<= a few hundred KB): re-send it with every call instead of tracking caller-side changes
  check(cudaMemcpyAsync(d_hk, hk_host, bank_elems * sizeof(float), cudaMemcpyHostToDevice, ws.st[0]));
  if (n_tab) check(cudaMemcpyAsync(d_tab, tables_host, (size_t)n_tab * sizeof(float), cudaMemcpyHostToDevice, ws.st[0]));
  check(cudaEventRecord(ws.bank_up, ws.st[0]));
  for (int i = 0; i < n_slots; ++i) check(cudaStreamWaitEvent(ws.kst[i], ws.bank_up, 0));  // no host-side wait: the first H2D copy follows at once
  // Chunk schedule: host_chunks / host_next_chunk above.
  // Copy phase: WHEN a D2H copy starts relative to the H2D copy running beside it decides what both directions get.  With the same
  // sixteen 16 MiB copies each way and only a delay between a chunk's H2D and its D2H (tools/e2e_pipeline_probe.py), a round trip takes
  // 5.87 ms at delay 0, 6.3 - 6.7 ms when the D2H starts 5 - 65 % into the next H2D copy, ~6.0 ms at 80 - 95 % and 6.2 - 6.8 ms again
  // from 100 % on.  A chunk's own D2H, issued behind its kernels, starts a kernel pair's latency (~30 us = 10 %) into the next H2D:
  // the bad zone.  So the copies get streams of their own in which the D2H of chunk i - 1 directly follows the H2D of chunk i (it starts
  // the instant that copy ends, i.e. together with the H2D of chunk i + 1), and the kernels run on separate streams, tied in by events:
  //   copy stream of chunk i  :  [kernels(i - n_slots) done]  H2D(i)  ->up(i)   [kernels(i - 1) done]  D2H(i - 1)  ->down(i - 1)
  //   kernel stream of chunk i:  [up(i)]  [down(i - n_slots)]  analysis(i), synthesis(i)  ->kdone(i)
  struct Pending {
    bool live = false;
    int slot = 0;
    long r0 = 0;
    size_t n = 0;
  } prev;
  auto copy_out = [&](const Pending& c, cudaStream_t s) {  // sub-bands and output of chunk c back to the host, once its kernels are done
    check(cudaStreamWaitEvent(s, ws.kdone[c.slot], 0));
    if (y_host) check(cudaMemcpyAsync(y_host + (size_t)c.r0 * clip_samples, ws.d_y[c.slot], c.n * sizeof(float), cudaMemcpyDeviceToHost, s));
    check(cudaMemcpyAsync(out_host + (size_t)c.r0 * clip_samples, ws.d_o[c.slot], c.n * sizeof(Sample), cudaMemcpyDeviceToHost, s));
    check(cudaEventRecord(ws.down[c.slot], s));
  };
  int slot = 0;
  long clips = 0, index = 0;
  for (long r0 = 0; r0 < B && rc == PQMF_OK; r0 += clips, slot = (slot + 1) % n_slots, ++index) {
    clips = host_next_chunk(plan, B, r0);
    const size_t n = (size_t)clips * clip_samples;
    cudaStream_t cs = ws.st[slot], ks = ws.kst[slot];
    const bool reused = index >= n_slots;
    if (reused) check(cudaStreamWaitEvent(cs, ws.kdone[slot], 0));  // the slot's previous kernels have read d_x
    check(cudaMemcpyAsync(ws.d_x[slot], x_host + (size_t)r0 * clip_samples, n * sizeof(Sample), cudaMemcpyHostToDevice, cs));
    check(cudaEventRecord(ws.up[slot], cs));
    if (prev.live) copy_out(prev, cs);
    prev.live = false;
    if (rc) break;
    check(cudaStreamWaitEvent(ks, ws.up[slot], 0));
    if (reused) check(cudaStreamWaitEvent(ks, ws.down[slot], 0));   // the slot's previous sub-bands / output have been copied out
    if (rc) break;
    if constexpr (kPcm) {
      rc = pqmf_analysis_pcm16(static_cast<const int16_t*>(ws.d_x[slot]), ws.d_y[slot], d_hk, d_tab, (int)clips, T, C, 0, F, M, L, flags, ks);
      if (rc) break;
      rc = pqmf_synthesis_pcm16(ws.d_y[slot], static_cast<int16_t*>(ws.d_o[slot]), d_hk, d_tab, (int)clips, C, F, M, L, delay_frames, flags, ks);
    } else {
      rc = pqmf_analysis_f32(static_cast<const float*>(ws.d_x[slot]), ws.d_y[slot], d_hk, d_tab, (int)clips, T, F, M, L, flags, ks);
      if (rc) break;
      rc = pqmf_synthesis_f32(ws.d_y[slot], static_cast<float*>(ws.d_o[slot]), d_hk, d_tab, (int)clips, F, M, L, delay_frames, flags, ks);
    }
    if (rc) break;
    check(cudaEventRecord(ws.kdone[slot], ks));
    prev.live = true;
    prev.slot = slot;
    prev.r0 = r0;
    prev.n = n;
  }
  if (prev.live && rc == PQMF_OK) copy_out(prev, ws.kst[prev.slot]);  // the last chunk: straight behind its kernels
  for (int i = 0; i < kHostSlots; ++i) {
    check(cudaStreamSynchronize(ws.st[i]));
    check(cudaStreamSynchronize(ws.kst[i]));
  }
  return rc;
}

// ---- stream pools.  The indexed Hankel-4 kernels exactly where a lockstep call with B = n runs the Hankel-4 streaming kernels (the
//      routing decision of h4_*_stream); the indexed direct form everywhere else -- including few-stream n_band 16, where a lockstep
//      call runs the fold kernels ----
int pool_analysis(const float* x, float* y, const float* hk, const float* tables, float* xpool, const PoolRows& pool, int n, long T, int M, int L,
                  unsigned flags, cudaStream_t st) {
  if (h4_analysis_stream(x, y, tables, xpool, xpool, n, T, M, L, 0, flags, st, &pool) == 0) {
    ++g_launches;
    return 0;
  }
  return analysis_direct(x, xpool, y, hk, n, T, T / M, M, L, L, 0, 0, st, pqmf::PcmIn{nullptr, 1, 0}, xpool, &pool);
}
int pool_synthesis(const float* s, float* out, const float* hk, const float* tables, float* spool, const PoolRows& pool, int n, long F, int M, int L,
                   unsigned flags, cudaStream_t st) {
  if (h4_synthesis_stream(s, out, tables, spool, spool, n, F, M, L, 0, flags, st, &pool) == 0) {
    ++g_launches;
    return 0;
  }
  return synthesis_direct(s, spool, out, hk, n, F, M, L, -M, 0, 0, st, nullptr, 1, nullptr, spool, &pool);
}
// after the compute launches of a call: flip the half and advance the parity of every listed stream (one launch on the same stream)
int pool_phase(const PoolRows& pool, int n, int* xphase, long x_frames, int* sphase, long s_frames, cudaStream_t st) {
  pqmf::stream_pool_phase_kernel<<<(n + 255) / 256, 256, 0, st>>>(pool.ids, n, pool.P, xphase, (int)(x_frames & 1), sphase, (int)(s_frames & 1));
  ++g_launches;
  return cuda_status();
}
bool bad_pool(int P, int n) { return P < 1 || n < 0 || n > P; }

}  // namespace

extern "C" {

int pqmf_abi_version(void) { return PQMF_B200_ABI_VERSION; }

const char* pqmf_strerror(int code) {
  switch (code) {
    case PQMF_OK: return "ok";
    case PQMF_ERR_ARG: return "pqmf_b200: invalid argument (null pointer, bad size or misaligned buffer)";
    case PQMF_ERR_UNSUPPORTED: return "pqmf_b200: unsupported parameter combination";
    case PQMF_ERR_NO_DEVICE: return "pqmf_b200: no usable CUDA device (needs sm_100)";
    default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "pqmf_b200: unknown error";
  }
}

unsigned long long pqmf_launch_count(void) { return g_launches.load(); }

int pqmf_path_for(int M, int L, const float* tables, unsigned flags) {
  return (use_fast(M, L, tables, flags) || use_h4_family(M, L, tables, flags)) ? 1 : 0;
}

long pqmf_tables_numel(int M, int L) {
  if (pqmf::hankel16_supported(M, L)) return kH4PairOffset + 2L * kH4PairImageFloats;
  return h4_family(M, L) ? h4_tables_floats(M, L) : 0;
}

int pqmf_build_tables_f32(const float* hk_host, const float* h_host, int N, int M, int L, float* tables_host,
                          double* residual, unsigned* fast_flags) {
  if (!hk_host || !h_host || !tables_host || N <= 0 || N > L) return PQMF_ERR_ARG;
  if (!pqmf::hankel16_supported(M, L)) {
    if (!h4_family(M, L)) return PQMF_ERR_UNSUPPORTED;
    // ---- other band counts / prototype lengths: CTA-pair images of the offline Hankel kernels only.  Taps kept = the span of
    //      non-zero columns rounded to the alignment the kernels need (32 for the flag fields, n_band for whole synthesis lags).
    int first = L, last = -1;
    for (int k = 0; k < M; ++k)
      for (int j = 0; j < L; ++j)
        if (hk_host[(size_t)k * L + j] != 0.f) {
          first = j < first ? j : first;
          last = j > last ? j : last;
        }
    if (last < 0) return PQMF_ERR_UNSUPPORTED;
    const int al = M > 32 ? M : 32;
    int jlo = (first / al) * al, kt = ((last + al) / al) * al - jlo;
    auto fits = [&](int j0, int k0) {
      return pqmf::h4_shape_fits(pqmf::h4_shape(M, j0, k0, true, false)) && pqmf::h4_shape_fits(pqmf::h4_shape(M, j0, k0, true, true));
    };
    bool split = false;
    if (!fits(jlo, kt)) {  // too long for one SM's shared memory: two tap ranges of equal length, two launches
      if (kt % (2 * al) != 0) {
        if (jlo + kt + al <= L) kt += al;
        else if (jlo >= al) { jlo -= al; kt += al; }
        else return PQMF_ERR_UNSUPPORTED;
      }
      kt /= 2;
      split = true;
      if (!fits(jlo, kt) || !fits(jlo + kt, kt) || h4_ks(M, kt) > h4_ks(M, L / 2)) return PQMF_ERR_UNSUPPORTED;
    }
    if (jlo / 32 > 15 || kt / 32 > 31) return PQMF_ERR_UNSUPPORTED;
    std::memset(tables_host, 0, (size_t)pqmf_tables_numel(M, L) * sizeof(float));
    uint16_t* base = reinterpret_cast<uint16_t*>(tables_host);
    const int ks = h4_ks(M, kt);
    std::vector<uint16_t> ia((size_t)2 * ks * 128 * 8), is((size_t)2 * ks * 128 * 8);
    if (!split) {
      pqmf::hankel4_build_banks(hk_host, M, L, jlo, kt, ia.data(), is.data());
      pqmf::hankel4_pair_image(ia.data(), ks, base);
      pqmf::hankel4_pair_image(is.data(), ks, base + 2 * h4_pair_floats(M, L));
      if (M < 8) {  // the synthesis image with one more (all-zero) lag at the top, see h4_pair_floats
        const int ks1 = h4_ks(M, kt + M);
        std::vector<uint16_t> ia1((size_t)2 * ks1 * 128 * 8), is1((size_t)2 * ks1 * 128 * 8);
        pqmf::hankel4_build_banks(hk_host, M, L, jlo, kt + M, ia1.data(), is1.data());
        pqmf::hankel4_pair_image(is1.data(), ks1, base + 2 * (2 * h4_pair_floats(M, L)));
      }
    } else {
      for (int half = 0; half < 2; ++half) {
        pqmf::hankel4_build_banks(hk_host, M, L, jlo + half * kt, kt, ia.data(), is.data());
        pqmf::hankel4_pair_image(ia.data(), ks, base + 2 * (half * h4_half_floats(M, L)));
        pqmf::hankel4_pair_image(is.data(), ks, base + 2 * ((2 + half) * h4_half_floats(M, L)));
      }
    }
    const int kt_all = split ? 2 * kt : kt;
    // long banks have long tails: the analysis field holds up to 31 steps per side (n_band 32: 9, n_band 64: 16 of 48 per tap range)
    const int trim_a = pqmf::hankel4_pick_trim(hk_host, M, L, jlo, kt_all, false, kTrimBudgetAnalysis, ks - 1 < 31 ? ks - 1 : 31);
    const int trim_s = pqmf::hankel4_pick_trim(hk_host, M, L, jlo, kt_all, true, kTrimBudgetSynthesis);
    if (residual) *residual = 0.0;
    if (fast_flags) *fast_flags = PQMF_FLAG_TAPS(jlo / 32, kt / 32) | PQMF_FLAG_H4_TRIM(trim_a, trim_s) | (split ? PQMF_FLAG_H4_SPLIT : 0u);
    return PQMF_OK;
  }
  std::memset(tables_host, 0, (size_t)pqmf_tables_numel(M, L) * sizeof(float));
  // ---- part 1: fold + modulation tables  [ g (L) | c1 (M*2M) | c2 (M*2M) ]
  // hk[k, r + 2M q] = (-1)^q * 2 hpad[r + 2M q] * cos((2k+1) pi/(2M) (r - c0) + (-1)^k pi/4)   (SURVEY.md A.3)
  //                 =  g[r + 2M q]              * C[k, r]
  const int pad_l = (L - N) / 2;       // center_pad_next_pow_2, reference pqmf.py:26-32
  const int c0 = pad_l + N / 2;        // column of the prototype centre
  const int R = 2 * M;
  float* g = tables_host;
  float* chi = tables_host + L;
  float* clo = chi + (size_t)M * R;
  for (int j = 0; j < L; ++j) {
    const int t = j - pad_l;
    const float hv = (t >= 0 && t < N) ? h_host[t] : 0.f;
    g[j] = ((j / R) & 1) ? -hv : hv;
  }
  const double pi = 3.14159265358979323846;
  std::vector<double> C((size_t)M * R);
  for (int k = 0; k < M; ++k)
    for (int r = 0; r < R; ++r)
      C[(size_t)k * R + r] = 2.0 * std::cos((2 * k + 1) * pi / (2.0 * M) * (r - c0) + ((k & 1) ? -pi / 4 : pi / 4));
  // two-term fp16 split of the modulation matrix: C = c1 + c2 (both exactly representable in fp16)
  for (size_t i = 0; i < (size_t)M * R; ++i) {
    const float hi = __half2float(__float2half_rn((float)C[i]));
    chi[i] = hi;
    clo[i] = __half2float(__float2half_rn((float)(C[i] - (double)hi)));
  }
  double res = 0.0;
  for (int k = 0; k < M; ++k)
    for (int j = 0; j < L; ++j) {
      const double model = (double)g[j] * C[(size_t)k * R + (j % R)];
      res = std::fmax(res, std::fabs((double)hk_host[(size_t)k * L + j] - model));
    }
  if (residual) *residual = res;
  // taps that are pure centre padding: with N = 377 of 512 the first and last 64 columns of hk are zero
  bool trimmed = true;
  for (int k = 0; k < M && trimmed; ++k)
    for (int j = 0; j < L; ++j)
      if ((j < 64 || j >= 448) && hk_host[(size_t)k * L + j] != 0.f) {
        trimmed = false;
        break;
      }
  for (int j = 0; j < L; ++j)
    if ((j < 64 || j >= 448) && g[j] != 0.f) trimmed = false;
  // ---- part 2: fp16 images of hk itself for the exact tensor-core path (hankel16.cuh)
  const int jlo = trimmed ? 64 : 0, kt = trimmed ? 384 : 512;
  uint16_t* img = reinterpret_cast<uint16_t*>(tables_host + kFoldTableFloats);
  pqmf::hankel16_build_banks(hk_host, jlo, kt, img, img + (size_t)kt * 32);
  // ---- part 3: the same bank replicated at four frame offsets for the offline default path (hankel4.cuh)
  uint16_t* img4 = reinterpret_cast<uint16_t*>(tables_host + kH4TableOffset);
  pqmf::hankel4_build_banks(hk_host, 16, 512, jlo, kt, img4, img4 + 2 * kH4ImageFloats);
  const int ks4 = (kt + 64 - 16 + 15) / 16;
  uint16_t* imgp = reinterpret_cast<uint16_t*>(tables_host + kH4PairOffset);
  pqmf::hankel4_pair_image(img4, ks4, imgp);
  pqmf::hankel4_pair_image(img4 + 2 * kH4ImageFloats, ks4, imgp + 2 * kH4PairImageFloats);
  // edge K-steps of the Hankel-4 kernels that may skip the fp16 correction terms (budgets: kTrimBudget*)
  const int trim_a = pqmf::hankel4_pick_trim(hk_host, 16, 512, jlo, kt, false, kTrimBudgetAnalysis);
  const int trim_s = pqmf::hankel4_pick_trim(hk_host, 16, 512, jlo, kt, true, kTrimBudgetSynthesis);
  if (fast_flags) *fast_flags = PQMF_FLAG_TAPS(jlo / 32, kt / 32) | PQMF_FLAG_H4_TRIM(trim_a, trim_s);
  return PQMF_OK;
}

int pqmf_analysis_f32(const float* x, float* y, const float* hk, const float* tables, int B, long T, long n_frames, int M,
                      int L, unsigned flags, pqmf_stream_t stream) {
  if (bad_dims(B, T, M, L) || n_frames < 0) return PQMF_ERR_ARG;
  if (B == 0 || n_frames == 0) return PQMF_OK;
  if (!x || !y || !hk) return PQMF_ERR_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  if (h4_route_analysis(B, T, n_frames, M, L, tables, flags) && h4_aligned_f32(x, y)) {
    int e = h4_analysis(x, y, tables, B, T, n_frames, M, L, flags, st);
    if (e != PQMF_ERR_UNSUPPORTED) { g_launches += (e == 0); return e; }
  }
  if (use_fast(M, L, tables, flags) && pqmf::hankel16_analysis_ok(x, y, T, n_frames)) {
    int e = fast_analysis(x, nullptr, y, nullptr, tables, B, T, n_frames, L / 2, 0, flags, st);
    if (e != PQMF_ERR_UNSUPPORTED) { g_launches += (e == 0); return e; }
  }
  return analysis_direct(x, nullptr, y, hk, B, T, n_frames, M, L, L / 2, 0, (flags & PQMF_FLAG_NO_SIGN) ? 1 : 0, st);
}

int pqmf_synthesis_f32(const float* s, float* out, const float* hk, const float* tables, int B, long n_frames, int M, int L,
                       int delay_frames, unsigned flags, pqmf_stream_t stream) {
  if (bad_dims(B, n_frames, M, L) || delay_frames < 0 || delay_frames > 1) return PQMF_ERR_ARG;
  if (B == 0 || n_frames == 0) return PQMF_OK;
  if (!s || !out || !hk) return PQMF_ERR_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  const int off2 = L / 2 - delay_frames * M;
  if (h4_route_synthesis(B, n_frames, M, L, tables, flags) && h4_aligned_f32(out, s)) {
    int e = h4_synthesis(s, out, tables, B, n_frames, off2, M, L, flags, st);
    if (e != PQMF_ERR_UNSUPPORTED) { g_launches += (e == 0); return e; }
  }
  if (use_fast(M, L, tables, flags) && pqmf::hankel16_synthesis_ok(s, out, n_frames)) {
    int e = fast_synthesis(s, nullptr, out, nullptr, tables, B, n_frames, off2, 0, flags, st);
    if (e != PQMF_ERR_UNSUPPORTED) { g_launches += (e == 0); return e; }
  }
  return synthesis_direct(s, nullptr, out, hk, B, n_frames, M, L, off2, 0, (flags & PQMF_FLAG_NO_SIGN) ? 1 : 0, st);
}

int pqmf_analysis_pcm16(const int16_t* pcm, float* y, const float* hk, const float* tables, int B, long T, int C, int downmix,
                        long n_frames, int M, int L, unsigned flags, pqmf_stream_t stream) {
  if (bad_dims(B, T, M, L) || n_frames < 0 || C < 1 || C > 64) return PQMF_ERR_ARG;
  const long rows = downmix ? (long)B : (long)B * C;
  if (rows >= (1L << 31)) return PQMF_ERR_ARG;
  if (B == 0 || n_frames == 0) return PQMF_OK;
  if (!pcm || !y || !hk) return PQMF_ERR_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  const pqmf::PcmIn in{pcm, C, downmix ? 1 : 0};
  if (use_h4_family(M, L, tables, flags) && use_h4((int)rows, n_frames, M, nullptr) && T > 0 && (T % M) == 0 && (T % 8) == 0 && n_frames == T / M &&
      ((uintptr_t)pcm % 32) == 0 && ((uintptr_t)y % 16) == 0) {
    const int e = h4_analysis(nullptr, y, tables, (int)rows, T, n_frames, M, L, flags, st, in);
    if (e != PQMF_ERR_UNSUPPORTED) { g_launches += (e == 0); return e; }
  }
  return analysis_direct(nullptr, nullptr, y, hk, (int)rows, T, n_frames, M, L, L / 2, 0, (flags & PQMF_FLAG_NO_SIGN) ? 1 : 0, st, in);
}

int pqmf_synthesis_pcm16(const float* s, int16_t* pcm, const float* hk, const float* tables, int B, int C, long n_frames, int M, int L,
                         int delay_frames, unsigned flags, pqmf_stream_t stream) {
  if (bad_dims(B, n_frames, M, L) || delay_frames < 0 || delay_frames > 1 || C < 1 || C > 64) return PQMF_ERR_ARG;
  const long rows = (long)B * C;
  if (rows >= (1L << 31)) return PQMF_ERR_ARG;
  if (B == 0 || n_frames == 0) return PQMF_OK;
  if (!s || !pcm || !hk) return PQMF_ERR_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  const int off2 = L / 2 - delay_frames * M;
  if (use_h4_family(M, L, tables, flags) && use_h4((int)rows, n_frames, M, nullptr) && n_frames > 0 && (n_frames & 3) == 0 && ((uintptr_t)s % 16) == 0 &&
      ((uintptr_t)pcm % 16) == 0) {
    const int e = h4_synthesis(s, nullptr, tables, (int)rows, n_frames, off2, M, L, flags, st, pcm, C);
    if (e != PQMF_ERR_UNSUPPORTED) { g_launches += (e == 0); return e; }
  }
  return synthesis_direct(s, nullptr, nullptr, hk, (int)rows, n_frames, M, L, off2, 0, (flags & PQMF_FLAG_NO_SIGN) ? 1 : 0, st, pcm, C);
}

int pqmf_synthesis_bands_f32(const float* const* bands, const long* lens, float* out, const float* hk, int B, long n_frames, int M, int L,
                             int delay_frames, const float* prev_tail, const float* fade_out, const float* fade_in, float* tail_out, int Lx,
                             unsigned flags, pqmf_stream_t stream) {
  if (bad_dims(B, n_frames, M, L) || delay_frames < 0 || delay_frames > 1 || M > pqmf::kMaxBandTable || Lx < 0) return PQMF_ERR_ARG;
  if (!bands || !lens) return PQMF_ERR_ARG;
  const bool fade = prev_tail != nullptr && Lx > 0;
  if (fade && (!fade_out || !fade_in || !tail_out || tail_out == prev_tail)) return PQMF_ERR_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  pqmf::BandTable t{};
  t.enabled = 1;
  t.Lx = Lx;
  for (int k = 0; k < M; ++k) {
    if (lens[k] < 0 || lens[k] >= (1L << 31) || (!bands[k] && lens[k] > 0 && B > 0)) return PQMF_ERR_ARG;
    t.band[k] = bands[k];
    t.len[k] = (int)lens[k];
    // centre crop / zero pad to n_frames (1-PitchShifterWrapper.py:279-289): cur > target: start = (cur - target) // 2; else left = pad // 2
    t.start[k] = lens[k] > n_frames ? (int)((lens[k] - n_frames) / 2) : -(int)((n_frames - lens[k]) / 2);
  }
  // the reference cross-fades only for batch 1 (:262); other batch sizes leave the bands and the kept tail as they are
  if (fade && B == 1) {
    t.prev_tail = prev_tail;
    t.fade_out = fade_out;
    t.fade_in = fade_in;
    const int n = M * Lx;
    pqmf::band_tail_kernel<<<(n + 255) / 256, 256, 0, st>>>(t, M, tail_out);
    ++g_launches;
    if (int e = cuda_status()) return e;
  } else if (fade) {
    cudaError_t e = cudaMemcpyAsync(tail_out, prev_tail, (size_t)M * Lx * sizeof(float), cudaMemcpyDeviceToDevice, st);
    if (e != cudaSuccess) return (int)e;
  }
  if (B == 0 || n_frames == 0) return PQMF_OK;
  if (!out || !hk) return PQMF_ERR_ARG;
  return synthesis_direct(nullptr, nullptr, out, hk, B, n_frames, M, L, L / 2 - delay_frames * M, 0, (flags & PQMF_FLAG_NO_SIGN) ? 1 : 0, st, nullptr, 1, &t);
}

int pqmf_analysis_stream_f32(const float* x, float* y, const float* hk, const float* tables, const float* state_in,
                             float* state_out, int B, long T, int M, int L, int frame_parity, unsigned flags,
                             pqmf_stream_t stream) {
  if (bad_dims(B, T, M, L) || (T % M) != 0) return PQMF_ERR_ARG;
  if (B == 0) return PQMF_OK;
  if (!hk || !state_in || !state_out || state_in == state_out) return PQMF_ERR_ARG;
  if (T == 0) return PQMF_ERR_ARG;
  if (!x || !y) return PQMF_ERR_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  const long F = T / M;
  // many streams: the streaming Hankel-4 kernels (n_band 8 / 16 / 32); few n_band-16 streams: the fold kernels
  if (h4_analysis_stream(x, y, tables, state_in, state_out, B, T, M, L, frame_parity, flags, st) == 0) { ++g_launches; return 0; }
  if (use_fast(M, L, tables, flags) && pqmf::hankel16_analysis_ok(x, y, T, F)) {
    int e = fast_analysis(x, state_in, y, state_out, tables, B, T, F, L, frame_parity & 1, flags, st);
    if (e != PQMF_ERR_UNSUPPORTED) { g_launches += (e == 0); return e; }
  }
  // fp32 direct form; the CTA of each row's last frame tile also rolls that row's history (no separate launch)
  return analysis_direct(x, state_in, y, hk, B, T, F, M, L, L, frame_parity, 0, st, pqmf::PcmIn{nullptr, 1, 0}, state_out);
}

int pqmf_synthesis_stream_f32(const float* s, float* out, const float* hk, const float* tables, const float* state_in,
                              float* state_out, int B, long n_frames, int M, int L, int frame_parity, unsigned flags,
                              pqmf_stream_t stream) {
  if (bad_dims(B, n_frames, M, L) || (L % M) != 0) return PQMF_ERR_ARG;
  if (B == 0) return PQMF_OK;
  if (!hk || !state_in || !state_out || state_in == state_out || n_frames == 0) return PQMF_ERR_ARG;
  if (!s || !out) return PQMF_ERR_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  const int K = L / M;
  // history frames sit K frames before frame 0 of the block: their parity offset is (frame_parity - K)
  if (h4_synthesis_stream(s, out, tables, state_in, state_out, B, n_frames, M, L, frame_parity, flags, st) == 0) { ++g_launches; return 0; }
  if (use_fast(M, L, tables, flags) && pqmf::hankel16_synthesis_ok(s, out, n_frames)) {
    int e = fast_synthesis(s, state_in, out, state_out, tables, B, n_frames, -M, frame_parity & 1, flags, st);
    if (e != PQMF_ERR_UNSUPPORTED) { g_launches += (e == 0); return e; }
  }
  return synthesis_direct(s, state_in, out, hk, B, n_frames, M, L, -M, frame_parity, 0, st, nullptr, 1, nullptr, state_out);
}

int pqmf_stream_step_f32(const float* x, float* y, float* out, const float* hk, const float* tables, const float* xstate_in, float* xstate_out,
                         const float* sstate_in, float* sstate_out, int B, long T, int M, int L, int parity_in, int parity_out, unsigned flags,
                         pqmf_stream_t stream) {
  if (bad_dims(B, T, M, L) || (T % M) != 0 || T == 0) return PQMF_ERR_ARG;
  if (B == 0) return PQMF_OK;
  if (!x || !y || !out || !hk || !xstate_in || !xstate_out || !sstate_in || !sstate_out || xstate_in == xstate_out || sstate_in == sstate_out)
    return PQMF_ERR_ARG;
  // Two launches on the same stream.  (One persistent kernel for both phases was built and measured: bit-identical and no faster,
  // experiments/fused_stream_step.cuh.txt -- the launches are not what a block step costs.)
  int e = pqmf_analysis_stream_f32(x, y, hk, tables, xstate_in, xstate_out, B, T, M, L, parity_in, flags, stream);
  if (e) return e;
  return pqmf_synthesis_stream_f32(y, out, hk, tables, sstate_in, sstate_out, B, T / M, M, L, parity_out, flags, stream);
}

int pqmf_stream_pool_analysis_f32(const float* x, float* y, const float* hk, const float* tables, float* xpool, int* xphase, int P,
                                  const int* ids, int n, long T, int M, int L, unsigned flags, pqmf_stream_t stream) {
  if (bad_dims(n, T, M, L) || bad_pool(P, n) || T <= 0 || (T % M) != 0) return PQMF_ERR_ARG;
  if (n == 0) return PQMF_OK;
  if (!x || !y || !hk || !xpool || !xphase || !ids) return PQMF_ERR_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  const PoolRows pool{ids, xphase, P};
  if (int e = pool_analysis(x, y, hk, tables, xpool, pool, n, T, M, L, flags, st)) return e;
  return pool_phase(pool, n, xphase, T / M, nullptr, 0, st);
}

int pqmf_stream_pool_synthesis_f32(const float* s, float* out, const float* hk, const float* tables, float* spool, int* sphase, int P,
                                   const int* ids, int n, long n_frames, int M, int L, unsigned flags, pqmf_stream_t stream) {
  if (bad_dims(n, n_frames, M, L) || bad_pool(P, n) || n_frames <= 0 || (L % M) != 0) return PQMF_ERR_ARG;
  if (n == 0) return PQMF_OK;
  if (!s || !out || !hk || !spool || !sphase || !ids) return PQMF_ERR_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  const PoolRows pool{ids, sphase, P};
  if (int e = pool_synthesis(s, out, hk, tables, spool, pool, n, n_frames, M, L, flags, st)) return e;
  return pool_phase(pool, n, nullptr, 0, sphase, n_frames, st);
}

int pqmf_stream_pool_step_f32(const float* x, float* y, float* out, const float* hk, const float* tables, float* xpool, int* xphase,
                              float* spool, int* sphase, int P, const int* ids, int n, long T, int M, int L, unsigned flags,
                              pqmf_stream_t stream) {
  if (bad_dims(n, T, M, L) || bad_pool(P, n) || T <= 0 || (T % M) != 0 || (L % M) != 0) return PQMF_ERR_ARG;
  if (n == 0) return PQMF_OK;
  if (!x || !y || !out || !hk || !xpool || !xphase || !spool || !sphase || !ids || xphase == sphase) return PQMF_ERR_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  const PoolRows xrows{ids, xphase, P}, srows{ids, sphase, P};
  if (int e = pool_analysis(x, y, hk, tables, xpool, xrows, n, T, M, L, flags, st)) return e;
  if (int e = pool_synthesis(y, out, hk, tables, spool, srows, n, T / M, M, L, flags, st)) return e;
  return pool_phase(xrows, n, xphase, T / M, sphase, T / M, st);
}

// ---- int16 PCM blocks in the streaming calls: the streaming Hankel-4 kernels with PCM loads (any channel count, optional down-mix) and
//      mono PCM stores, exactly where the fp32 call with the same rows runs those kernels (h4_*_stream_ok, with the PCM buffer's alignment);
//      every other call returns PQMF_ERR_UNSUPPORTED before anything is launched and the caller stages it through the fp32 entry ----
static bool pcm_args_bad(int C, long rows) { return C < 1 || C > 64 || rows >= (1L << 31); }

int pqmf_analysis_stream_pcm16(const int16_t* pcm, float* y, const float* hk, const float* tables, const float* state_in, float* state_out, int B,
                               long T, int C, int downmix, int M, int L, int frame_parity, unsigned flags, pqmf_stream_t stream) {
  const long rows = downmix ? (long)B : (long)B * C;
  if (bad_dims(B, T, M, L) || (T % M) != 0 || pcm_args_bad(C, rows)) return PQMF_ERR_ARG;
  if (B == 0) return PQMF_OK;
  if (!hk || !state_in || !state_out || state_in == state_out || T == 0 || !pcm || !y) return PQMF_ERR_ARG;
  const pqmf::PcmIn in{pcm, C, downmix ? 1 : 0};
  if (h4_analysis_stream(nullptr, y, tables, state_in, state_out, (int)rows, T, M, L, frame_parity, flags, (cudaStream_t)stream, nullptr, &in) != 0)
    return PQMF_ERR_UNSUPPORTED;  // nothing was launched
  ++g_launches;
  return PQMF_OK;
}

int pqmf_synthesis_stream_pcm16(const float* s, int16_t* pcm, const float* hk, const float* tables, const float* state_in, float* state_out, int B,
                                int C, long n_frames, int M, int L, int frame_parity, unsigned flags, pqmf_stream_t stream) {
  const long rows = (long)B * C;
  if (bad_dims(B, n_frames, M, L) || (L % M) != 0 || pcm_args_bad(C, rows)) return PQMF_ERR_ARG;
  if (B == 0) return PQMF_OK;
  if (!hk || !state_in || !state_out || state_in == state_out || n_frames == 0 || !s || !pcm) return PQMF_ERR_ARG;
  if (C != 1 ||
      h4_synthesis_stream(s, nullptr, tables, state_in, state_out, (int)rows, n_frames, M, L, frame_parity, flags, (cudaStream_t)stream, nullptr, pcm) != 0)
    return PQMF_ERR_UNSUPPORTED;
  ++g_launches;
  return PQMF_OK;
}

int pqmf_stream_step_pcm16(const int16_t* pcm, float* y, int16_t* pcm_out, const float* hk, const float* tables, const float* xstate_in,
                           float* xstate_out, const float* sstate_in, float* sstate_out, int B, long T, int C, int downmix, int M, int L, int parity_in,
                           int parity_out, unsigned flags, pqmf_stream_t stream) {
  const long rows = downmix ? (long)B : (long)B * C;
  if (bad_dims(B, T, M, L) || (T % M) != 0 || T == 0 || (L % M) != 0 || pcm_args_bad(C, rows)) return PQMF_ERR_ARG;
  if (B == 0) return PQMF_OK;
  if (!pcm || !y || !pcm_out || !hk || !xstate_in || !xstate_out || !sstate_in || !sstate_out || xstate_in == xstate_out ||
      sstate_in == sstate_out)
    return PQMF_ERR_ARG;
  // both directions native, or nothing is launched
  pqmf::H4AnalysisStreamParams pa{};
  pqmf::H4SynthesisStreamParams ps{};
  if ((downmix == 0 && C != 1) || !h4_analysis_stream_ok((int)rows, T, M, L, tables, flags, pcm, y, xstate_in, xstate_out, pa) ||
      !h4_synthesis_stream_ok((int)rows, T / M, M, L, tables, flags, y, pcm_out, true, sstate_in, sstate_out, ps))
    return PQMF_ERR_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  const pqmf::PcmIn in{pcm, C, downmix ? 1 : 0};
  if (h4_analysis_stream(nullptr, y, tables, xstate_in, xstate_out, (int)rows, T, M, L, parity_in, flags, st, nullptr, &in) != 0)
    return PQMF_ERR_UNSUPPORTED;  // the launch did not start: nothing ran
  ++g_launches;
  // the analysis has run: a failed synthesis launch is an error, not a refusal (a staged retry would step the analysis state twice)
  const int e = h4_synthesis_stream(y, nullptr, tables, sstate_in, sstate_out, (int)rows, T / M, M, L, parity_out, flags, st, nullptr, pcm_out);
  if (e != 0) return e > 0 ? e : (int)cudaErrorLaunchFailure;
  ++g_launches;
  return PQMF_OK;
}

int pqmf_stream_pool_analysis_pcm16(const int16_t* pcm, float* y, const float* hk, const float* tables, float* xpool, int* xphase, int P,
                                    const int* ids, int B, long T, int C, int downmix, int M, int L, unsigned flags, pqmf_stream_t stream) {
  const long rows = downmix ? (long)B : (long)B * C;
  if (bad_dims(B, T, M, L) || pcm_args_bad(C, rows) || bad_pool(P, (int)rows) || T <= 0 || (T % M) != 0) return PQMF_ERR_ARG;
  if (B == 0) return PQMF_OK;
  if (!pcm || !y || !hk || !xpool || !xphase || !ids) return PQMF_ERR_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  const PoolRows pool{ids, xphase, P};
  const pqmf::PcmIn in{pcm, C, downmix ? 1 : 0};
  if (h4_analysis_stream(nullptr, y, tables, xpool, xpool, (int)rows, T, M, L, 0, flags, st, &pool, &in) != 0) return PQMF_ERR_UNSUPPORTED;
  ++g_launches;
  return pool_phase(pool, (int)rows, xphase, T / M, nullptr, 0, st);
}

int pqmf_stream_pool_synthesis_pcm16(const float* s, int16_t* pcm, const float* hk, const float* tables, float* spool, int* sphase, int P,
                                     const int* ids, int B, int C, long n_frames, int M, int L, unsigned flags, pqmf_stream_t stream) {
  const long rows = (long)B * C;
  if (bad_dims(B, n_frames, M, L) || pcm_args_bad(C, rows) || bad_pool(P, (int)rows) || n_frames <= 0 || (L % M) != 0) return PQMF_ERR_ARG;
  if (B == 0) return PQMF_OK;
  if (!s || !pcm || !hk || !spool || !sphase || !ids) return PQMF_ERR_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  const PoolRows pool{ids, sphase, P};
  if (C != 1 || h4_synthesis_stream(s, nullptr, tables, spool, spool, (int)rows, n_frames, M, L, 0, flags, st, &pool, pcm) != 0)
    return PQMF_ERR_UNSUPPORTED;
  ++g_launches;
  return pool_phase(pool, (int)rows, nullptr, 0, sphase, n_frames, st);
}

int pqmf_stream_pool_step_pcm16(const int16_t* pcm, float* y, int16_t* pcm_out, const float* hk, const float* tables, float* xpool, int* xphase,
                                float* spool, int* sphase, int P, const int* ids, int B, long T, int C, int downmix, int M, int L, unsigned flags,
                                pqmf_stream_t stream) {
  const long rows = downmix ? (long)B : (long)B * C;
  if (bad_dims(B, T, M, L) || pcm_args_bad(C, rows) || bad_pool(P, (int)rows) || T <= 0 || (T % M) != 0 || (L % M) != 0) return PQMF_ERR_ARG;
  if (B == 0) return PQMF_OK;
  if (!pcm || !y || !pcm_out || !hk || !xpool || !xphase || !spool || !sphase || !ids || xphase == sphase) return PQMF_ERR_ARG;
  pqmf::H4AnalysisStreamParams pa{};
  pqmf::H4SynthesisStreamParams ps{};
  if ((downmix == 0 && C != 1) || !h4_analysis_stream_ok((int)rows, T, M, L, tables, flags, pcm, y, xpool, xpool, pa) ||
      !h4_synthesis_stream_ok((int)rows, T / M, M, L, tables, flags, y, pcm_out, true, spool, spool, ps))
    return PQMF_ERR_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  const PoolRows xrows{ids, xphase, P}, srows{ids, sphase, P};
  const pqmf::PcmIn in{pcm, C, downmix ? 1 : 0};
  if (h4_analysis_stream(nullptr, y, tables, xpool, xpool, (int)rows, T, M, L, 0, flags, st, &xrows, &in) != 0) return PQMF_ERR_UNSUPPORTED;
  ++g_launches;
  const int e = h4_synthesis_stream(y, nullptr, tables, spool, spool, (int)rows, T / M, M, L, 0, flags, st, &srows, pcm_out);
  if (e != 0) return e > 0 ? e : (int)cudaErrorLaunchFailure;  // see pqmf_stream_step_pcm16
  ++g_launches;
  return pool_phase(xrows, (int)rows, xphase, T / M, sphase, T / M, st);
}

int pqmf_roundtrip_f32(const float* x, float* y, float* out, const float* hk, const float* tables, int B, long T, long n_frames,
                       int M, int L, int delay_frames, unsigned flags, pqmf_stream_t stream) {
  if (bad_dims(B, T, M, L) || n_frames < 0 || delay_frames < 0 || delay_frames > 1) return PQMF_ERR_ARG;
  if (B == 0 || n_frames == 0) return PQMF_OK;
  if (!x || !y || !out || !hk) return PQMF_ERR_ARG;
  // One launch per direction over the whole batch.  Running the rows in chunks whose sub-bands fit the L2 (so that synthesis
  // never reads them from HBM) was measured at the bench shape and loses: 16 MB chunks -35 %, 32 MB -19 %, 64 MB -6 %, 128 MB
  // -2 % against the plain pair of launches -- every extra launch pays a pipeline fill and drain on all SMs.  What survives
  // is the hand-off built into the kernels: synthesis walks its tiles last-to-first and finds the tail of y in L2.
  int e = pqmf_analysis_f32(x, y, hk, tables, B, T, n_frames, M, L, flags, stream);
  if (e) return e;
  return pqmf_synthesis_f32(y, out, hk, tables, B, n_frames, M, L, delay_frames, flags, stream);
}

// rows per chunk of pqmf_reconstruct_f32: the chunk's sub-bands (rows * T * 4 bytes, 96 MB by default) are mostly still in the 126 MB L2
// when the synthesis launch of the chunk reads them, and a chunk is large enough for the tensor-core kernels (>= 96 tiles of 8192
// samples) whenever the batch is.  Measured at 64 x 2^20 against process() (tools/process_bench.py, sustained / burst): 32 MB chunks
// -13 % / -38 %, 48 MB -12 % / -27 %, 64 MB -6 % / -22 %, 96 MB -4 % / -13 %, 128 MB -2 % / -10 %: every extra launch pair costs a pipeline
// fill and drain on all SMs, so the chunk is as large as still saves most of the sub-band tensor (96 MB scratch instead of 268 MB).
long recon_chunk_rows(int B, long T) {
  static const long chunk_bytes = [] {
    const char* e = getenv("PQMF_RECON_CHUNK_MIB");   // tuning knob, read once
    const long v = e ? atol(e) : 0;
    return (v > 0 && v <= 4096 ? v : 96L) << 20;
  }();
  const long row_bytes = T * (long)sizeof(float);
  long rows = chunk_bytes / (row_bytes > 0 ? row_bytes : 1);
  const long tiles_per_row = (T + pqmf::kH4TileSamples - 1) / pqmf::kH4TileSamples;
  const long min_rows = (96 + tiles_per_row - 1) / (tiles_per_row > 0 ? tiles_per_row : 1);
  if (rows < min_rows) rows = min_rows;
  if (rows < 1) rows = 1;
  return rows < B ? rows : B;
}

size_t pqmf_reconstruct_scratch_bytes(int B, long T, long n_frames, int M) {
  if (B <= 0 || T <= 0 || n_frames <= 0 || M <= 0) return 0;
  return (size_t)recon_chunk_rows(B, T) * (size_t)M * (size_t)n_frames * sizeof(float);
}

int pqmf_reconstruct_f32(const float* x, float* out, float* scratch, size_t scratch_bytes, const float* hk, const float* tables, int B, long T,
                         long n_frames, int M, int L, int delay_frames, unsigned flags, pqmf_stream_t stream) {
  if (bad_dims(B, T, M, L) || n_frames < 0 || delay_frames < 0 || delay_frames > 1) return PQMF_ERR_ARG;
  if (B == 0 || n_frames == 0) return PQMF_OK;
  if (!x || !out || !hk || !scratch || scratch_bytes < pqmf_reconstruct_scratch_bytes(B, T, n_frames, M)) return PQMF_ERR_ARG;
  const long rows = recon_chunk_rows(B, T);
  for (long r0 = 0; r0 < B; r0 += rows) {
    const int n = (int)(B - r0 < rows ? B - r0 : rows);
    int e = pqmf_analysis_f32(x + (size_t)r0 * T, scratch, hk, tables, n, T, n_frames, M, L, flags, stream);
    if (e) return e;
    e = pqmf_synthesis_f32(scratch, out + (size_t)r0 * M * n_frames, hk, tables, n, n_frames, M, L, delay_frames, flags, stream);
    if (e) return e;
  }
  return PQMF_OK;
}

// ---- half-precision I/O: the offline Hankel-4 kernels with fp16 / bf16 loads and stores (half_io.cuh), wherever the fp32 call
//      would run them (h4_route_*); every other call is refused before anything is launched ----
int pqmf_analysis_x(const void* x, void* y, const float* hk, const float* tables, int B, long T, long n_frames, int M, int L, unsigned flags,
                    int dtype, pqmf_stream_t stream) {
  if (dtype == PQMF_DTYPE_F32)
    return pqmf_analysis_f32(static_cast<const float*>(x), static_cast<float*>(y), hk, tables, B, T, n_frames, M, L, flags, stream);
  pqmf::H4Io io;
  if (!half_io_of(dtype, io) || bad_dims(B, T, M, L) || n_frames < 0) return PQMF_ERR_ARG;
  if (B == 0 || n_frames == 0) return PQMF_OK;
  if (!x || !y || !hk) return PQMF_ERR_ARG;
  if (!half_analysis_native(x, y, B, T, n_frames, M, L, tables, flags)) return PQMF_ERR_UNSUPPORTED;
  const int e = h4_analysis(x, y, tables, B, T, n_frames, M, L, flags, (cudaStream_t)stream, pqmf::PcmIn{nullptr, 1, 0}, io);
  g_launches += (e == 0);
  return e;
}

int pqmf_synthesis_x(const void* s, void* out, const float* hk, const float* tables, int B, long n_frames, int M, int L, int delay_frames,
                     unsigned flags, int dtype, pqmf_stream_t stream) {
  if (dtype == PQMF_DTYPE_F32)
    return pqmf_synthesis_f32(static_cast<const float*>(s), static_cast<float*>(out), hk, tables, B, n_frames, M, L, delay_frames, flags, stream);
  pqmf::H4Io io;
  if (!half_io_of(dtype, io) || bad_dims(B, n_frames, M, L) || delay_frames < 0 || delay_frames > 1) return PQMF_ERR_ARG;
  if (B == 0 || n_frames == 0) return PQMF_OK;
  if (!s || !out || !hk) return PQMF_ERR_ARG;
  if (!half_synthesis_native(s, out, B, n_frames, M, L, tables, flags)) return PQMF_ERR_UNSUPPORTED;
  const int e = h4_synthesis(s, out, tables, B, n_frames, L / 2 - delay_frames * M, M, L, flags, (cudaStream_t)stream, nullptr, 1, io);
  g_launches += (e == 0);
  return e;
}

int pqmf_roundtrip_x(const void* x, void* y, void* out, const float* hk, const float* tables, int B, long T, long n_frames, int M, int L,
                     int delay_frames, unsigned flags, int dtype, pqmf_stream_t stream) {
  if (dtype == PQMF_DTYPE_F32)
    return pqmf_roundtrip_f32(static_cast<const float*>(x), static_cast<float*>(y), static_cast<float*>(out), hk, tables, B, T, n_frames, M, L,
                              delay_frames, flags, stream);
  pqmf::H4Io io;
  if (!half_io_of(dtype, io) || bad_dims(B, T, M, L) || n_frames < 0 || delay_frames < 0 || delay_frames > 1) return PQMF_ERR_ARG;
  if (B == 0 || n_frames == 0) return PQMF_OK;
  if (!x || !y || !out || !hk) return PQMF_ERR_ARG;
  // both directions native, or neither is launched
  if (!half_analysis_native(x, y, B, T, n_frames, M, L, tables, flags) || !half_synthesis_native(y, out, B, n_frames, M, L, tables, flags))
    return PQMF_ERR_UNSUPPORTED;
  const int e = pqmf_analysis_x(x, y, hk, tables, B, T, n_frames, M, L, flags, dtype, stream);
  if (e) return e;
  return pqmf_synthesis_x(y, out, hk, tables, B, n_frames, M, L, delay_frames, flags, dtype, stream);
}

// the sub-bands of a chunk are half-width here: the scratch sized for fp32 sub-bands holds them with room to spare
int pqmf_reconstruct_x(const void* x, void* out, void* scratch, size_t scratch_bytes, const float* hk, const float* tables, int B, long T,
                       long n_frames, int M, int L, int delay_frames, unsigned flags, int dtype, pqmf_stream_t stream) {
  if (dtype == PQMF_DTYPE_F32)
    return pqmf_reconstruct_f32(static_cast<const float*>(x), static_cast<float*>(out), static_cast<float*>(scratch), scratch_bytes, hk, tables, B, T,
                                n_frames, M, L, delay_frames, flags, stream);
  pqmf::H4Io io;
  if (!half_io_of(dtype, io) || bad_dims(B, T, M, L) || n_frames < 0 || delay_frames < 0 || delay_frames > 1) return PQMF_ERR_ARG;
  if (B == 0 || n_frames == 0) return PQMF_OK;
  if (!x || !out || !hk || !scratch || scratch_bytes < pqmf_reconstruct_scratch_bytes(B, T, n_frames, M)) return PQMF_ERR_ARG;
  const long rows = recon_chunk_rows(B, T);
  const uint16_t* xh = static_cast<const uint16_t*>(x);
  uint16_t* oh = static_cast<uint16_t*>(out);
  // every chunk native in both directions (a short last chunk may have too few tiles), or nothing is launched
  for (long r0 = 0; r0 < B; r0 += rows) {
    const int n = (int)(B - r0 < rows ? B - r0 : rows);
    if (!half_analysis_native(xh + (size_t)r0 * T, scratch, n, T, n_frames, M, L, tables, flags) ||
        !half_synthesis_native(scratch, oh + (size_t)r0 * M * n_frames, n, n_frames, M, L, tables, flags))
      return PQMF_ERR_UNSUPPORTED;
  }
  for (long r0 = 0; r0 < B; r0 += rows) {
    const int n = (int)(B - r0 < rows ? B - r0 : rows);
    int e = pqmf_analysis_x(xh + (size_t)r0 * T, scratch, hk, tables, n, T, n_frames, M, L, flags, dtype, stream);
    if (e) return e;
    e = pqmf_synthesis_x(scratch, oh + (size_t)r0 * M * n_frames, hk, tables, n, n_frames, M, L, delay_frames, flags, dtype, stream);
    if (e) return e;
  }
  return PQMF_OK;
}

int pqmf_roundtrip_host_f32(const float* x_host, float* y_host, float* out_host, const float* hk_host,
                            const float* tables_host, int B, long T, int M, int L, int delay_frames, unsigned flags,
                            int device) {
  return roundtrip_host(x_host, y_host, out_host, hk_host, tables_host, B, T, 1, M, L, delay_frames, flags, device);
}

int pqmf_roundtrip_host_pcm16(const int16_t* pcm_host, float* y_host, int16_t* out_host, const float* hk_host,
                              const float* tables_host, int B, long T, int C, int M, int L, int delay_frames, unsigned flags,
                              int device) {
  if (C < 1 || C > 64) return PQMF_ERR_ARG;
  return roundtrip_host(pcm_host, y_host, out_host, hk_host, tables_host, B, T, C, M, L, delay_frames, flags, device);
}

int pqmf_host_chunk_plan(int B, long T, int C, long* clips, int max_chunks) {
  if (B <= 0 || T <= 0 || C <= 0) return PQMF_ERR_ARG;
  const HostChunks plan = host_chunks(B, T, C);
  int n = 0;
  for (long r0 = 0; r0 < B; ++n) {
    const long c = host_next_chunk(plan, B, r0);
    if (clips && n < max_chunks) clips[n] = c;
    r0 += c;
  }
  return n;
}

void pqmf_shard_rows(long n_rows, int n_shards, int shard, long* start, long* count) {
  // contiguous, disjoint, covering; sizes differ by at most one (the same rule as pqmf_b200/sharding.py: shard_rows)
  const long base = n_shards > 0 ? n_rows / n_shards : 0, extra = n_shards > 0 ? n_rows % n_shards : 0;
  if (start) *start = (long)shard * base + (shard < extra ? shard : extra);
  if (count) *count = base + (shard < extra ? 1 : 0);
}

int pqmf_roundtrip_host_multi_f32(const float* x_host, float* y_host, float* out_host, const float* hk_host,
                                  const float* tables_host, int B, long T, int M, int L, int delay_frames, unsigned flags,
                                  const int* devices, int n_devices) {
  if (!devices || n_devices < 1 || n_devices > kMaxDevices) return PQMF_ERR_ARG;
  if (bad_dims(B, T, M, L) || !x_host || !out_host || !hk_host || (T % M) != 0) return PQMF_ERR_ARG;
  if (n_devices == 1) return pqmf_roundtrip_host_f32(x_host, y_host, out_host, hk_host, tables_host, B, T, M, L, delay_frames, flags, devices[0]);
  // rows are independent (SURVEY 8e): contiguous shards, sizes differing by at most one, one host thread per device, no collective
  std::vector<std::thread> workers;
  std::vector<int> rcs((size_t)n_devices, PQMF_OK);
  for (int i = 0; i < n_devices; ++i) {
    long r0 = 0, rows = 0;
    pqmf_shard_rows(B, n_devices, i, &r0, &rows);
    if (rows > 0) {
      const size_t off = (size_t)r0 * T;
      workers.emplace_back([=, &rcs] {
        rcs[(size_t)i] = pqmf_roundtrip_host_f32(x_host + off, y_host ? y_host + off : nullptr, out_host + off, hk_host, tables_host, (int)rows, T, M, L,
                                                 delay_frames, flags, devices[i]);
      });
    }
  }
  for (auto& w : workers) w.join();
  for (int rc : rcs)
    if (rc != PQMF_OK) return rc;
  return PQMF_OK;
}

void pqmf_host_release(void) {
  int cur = 0;
  cudaGetDevice(&cur);
  for (int d = 0; d < kMaxDevices; ++d) {
    HostWorkspace& ws = g_host_ws[d];
    std::lock_guard<std::mutex> lock(ws.mutex);
    if (!ws.streams_ready && !ws.d_bank && !ws.chunk_elems) continue;
    cudaSetDevice(d);
    for (int i = 0; i < kHostSlots; ++i) {
      if (ws.d_x[i]) cudaFree(ws.d_x[i]);
      if (ws.d_y[i]) cudaFree(ws.d_y[i]);
      if (ws.d_o[i]) cudaFree(ws.d_o[i]);
      if (ws.streams_ready && ws.st[i]) cudaStreamDestroy(ws.st[i]);
      if (ws.streams_ready && ws.kst[i]) cudaStreamDestroy(ws.kst[i]);
      if (ws.streams_ready && ws.up[i]) cudaEventDestroy(ws.up[i]);
      if (ws.streams_ready && ws.kdone[i]) cudaEventDestroy(ws.kdone[i]);
      if (ws.streams_ready && ws.down[i]) cudaEventDestroy(ws.down[i]);
    }
    if (ws.d_bank) cudaFree(ws.d_bank);
    if (ws.streams_ready && ws.bank_up) cudaEventDestroy(ws.bank_up);
    ws.bank_up = nullptr;
    for (int i = 0; i < kHostSlots; ++i) {
      ws.st[i] = ws.kst[i] = nullptr;
      ws.up[i] = ws.kdone[i] = ws.down[i] = nullptr;
      ws.d_x[i] = ws.d_o[i] = nullptr;
      ws.d_y[i] = nullptr;
    }
    ws.d_bank = nullptr;
    ws.chunk_elems = ws.bank_elems = 0;
    ws.streams_ready = false;
  }
  cudaSetDevice(cur);
}

}  // extern "C"
