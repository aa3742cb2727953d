// Offline PQMF for n_band 8 / 16 / 32 / 64: the direct form as an implicit-Hankel GEMM on the tensor cores, 64 samples per operand row.
// (n_band 64 and other banks too long for one SM's shared memory run as two tap ranges = two launches, the second accumulating.)
//
// hankel16.cuh shows that a strided signal can be fed to tcgen05.mma without im2col (one frame = 32 B = the SWIZZLE_32B row
// pitch), but there every 16 taps cost a full shared-memory read of the 128-row A tile (~111 B/sample: smem-bound at ~30 % of
// the HBM roofline).  Here one A row holds 64 samples = FR = 64 / M frames (128 B in fp16 = the SWIZZLE_128B row pitch; four
// frames at n_band 16, hence "Hankel-4") and the bank is replicated at the FR frame offsets along N, so N = FR * M * 2 = 128
// for every M:
//   analysis : D[i, (delta, k)] = sum_kappa X[64 i + kappa] * hk[k, kappa - M delta]               = y[k, frame FR i + delta]
//   synthesis: D[i, (delta, p)] = sum_(e,kb) S^T[FR i + e + n0, kb] * M hk[kb, M (delta + ehi - e) + p] = out[M (FR i + delta) + p]
// One 128-row MMA group yields 8192 samples; K-step s reads rows starting at byte 32 s of row i (128 (s / 4) + 32 (s % 4)).
// Precision: the same two-term fp16 split as hankel16.cuh (exact in hk up to 2^-22), columns 0-63 main term, 64-127 the
// c2 correction; the second pass (h2) uses only the c1 half (N = 64).  Edge K-steps whose correction terms are provably
// negligible for the actual bank run the main term only (h4_issue_mmas, hankel4_pick_trim).
// Roles: worker warps convert fp32 -> 2 x fp16 planes (swizzled STS) and drain TMEM; ONE warp only issues the MMAs
// (tcgen05.mma issue blocks the issuing thread while the tensor queue is full).  With PAIR the kernel runs as clusters of two
// CTAs sharing the bank operand (cta_group::2).  DESIGN.md section 5 has the measurements behind each of these choices.
// IO (half_io.cuh) is the sample format at the kernel's edge -- fp32, fp16 / bf16 (widened exactly in the loads, rounded to nearest
// even in the stores) or int16 PCM (pcm.cuh); everything between the loads and the stores is the same for all of them.
//
// Round 2: the second fp16 term of every sample and the second term of the bank are scaled by 2^11 (h2' = 2^11 (x - h1),
// c2' = 2^11 (2^10 hk - c1)) and accumulate in their own TMEM columns: D[:, 0:64] = h1 c1, D[:, 64:128] = h1 c2' + h2' c1, result =
// 2^-10 (D0 + 2^-11 D1).  Same MMA count, but the residuals stay in the fp16 normal range: the absolute error floor drops from 2^-25 to
// 2^-36 per sample.  The analysis window is loaded 8 samples (256 bits) at a time.
// Measured on one box against this file and NOT kept (bench.py's 20-step loop, medians of 4 alternating runs, DESIGN.md 5.7): the
// fp32 input staged in a shared-memory ring by bulk copies two tiles ahead (bit-identical, 7-9 % slower: shared-memory bandwidth is
// the binding resource -- the tensor pipe already reads ~250 KB of operands per tile); an L2 prefetch of the tile after next
// (cp.async.bulk.prefetch.L2: analysis -3 %, synthesis +14 %); three plane pairs / accumulators so the workers run two tiles ahead
// (+2 %): the board is power-capped during these kernels, extra activity costs clock.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <string.h>

#include <atomic>

#include "half_io.cuh"
#include "hankel16.cuh"
#include "pcm.cuh"
#include "ptx.cuh"

namespace pqmf {

constexpr int kH4Workers = 256;                 // analysis: convert + drain warps
constexpr int kH4Threads = kH4Workers + 32;     // + one warp that only issues tcgen05.mma
constexpr int kH4SynWorkers = 288;              // synthesis: nine worker warps, one (frame quad, band group) item per thread
constexpr int kH4SynThreads = kH4SynWorkers + 32;
constexpr int kH4Rows = 128;                    // A rows per tile
constexpr int kH4TileSamples = 64 * kH4Rows;    // 8192 samples (= 128 FR frames) per tile
constexpr int kH4MaxPlaneRows = 144;            // register prefetch / item counts are sized for this: K-steps <= 64
constexpr float kH4Res = 2048.0f;               // scale of the second fp16 term of samples and bank (2^11)

// K-major SWIZZLE_128B descriptor: rows 128 B apart, 8-row groups 1024 B apart, 16-byte chunk index ^= address bits 7-9
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024u >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
__device__ __forceinline__ uint32_t sw128_offset(uint32_t byte_lin) { return byte_lin ^ (((byte_lin >> 7) & 7u) << 4); }

// Shape of one launch (host and device).  PAIR: the kernel runs as a cluster of two CTAs (tcgen05 cta_group::2).  One M = 256
// MMA covers the two CTAs' tiles; each CTA holds only its half of the bank rows: rank 0 [c1 (64 rows) | c1 rows 0-31 again],
// rank 1 [c2 (64 rows) | c1 rows 32-63], i.e. rows 0-63 are this rank's half of the N = 128 operand and rows 64-95 its half of
// the N = 64 operand (at the same offset in both CTAs, because one descriptor addresses both).  Per SM and K-step the tensor
// pipe then reads 6 + 5 KB of operands instead of 8 + 6 KB (experiments/probe_h4_pair.cu).
struct H4Shape {
  int jlo, kt, ks;     // first non-zero tap, taps kept (multiples of 32), K-steps = ceil((kt + 64 - M) / 16)
  int rows, plane;     // 128-byte rows of one fp16 plane, bytes per plane (multiple of 1024)
  int bank;            // bytes of one CTA's bank image: [2 ks chunks][96 or 128 rows][16 B]
  int bytes;           // dynamic shared memory
};
inline H4Shape h4_shape(int M, int jlo, int kt, bool pair, bool synthesis, int extra_pad_bytes = 0) {
  H4Shape g;
  g.jlo = jlo;
  g.kt = kt;
  g.ks = (kt + 64 - M + 15) / 16;
  const int pad_bytes = (synthesis ? 3 * 2 * M : 0) + extra_pad_bytes;  // synthesis shifts its windows by up to 3 frames (alignment); streaming
                                                                        // blocks may shift theirs to make the history whole rows
  g.rows = kH4Rows + (32 * g.ks + pad_bytes - 1) / 128;
  g.plane = ((g.rows * 128 + 1023) / 1024) * 1024;
  g.bank = g.ks * 2 * (pair ? 96 : 128) * 16;
  g.bytes = g.bank + 4 * g.plane + 128;
  return g;
}
inline bool h4_shape_fits(const H4Shape& g) { return g.rows <= kH4MaxPlaneRows && g.bytes <= 227 * 1024; }

// one elected lane: the MMAs of a tile, D[:, 0:128] = h1 [c1 | c2']^T, D[:, 64:128] += h2' c1^T.  The first `tlo` and last `thi`
// K-steps carry only the tails of the prototype: there the two correction terms (h1 c2, h2 c1) are below the error budget
// that pqmf_build_tables_f32 checked against the actual bank, so those steps run h1 c1 alone (N = 64) and no h2 pass.
// (Issue order matters: all N = 128 MMAs, then all N = 64 ones -- alternating the two shapes was measured slower,
// experiments/probe_mma_order.cu.)
// `pad_bytes` shifts the A windows (synthesis alignment).
template <bool PAIR>
__device__ __forceinline__ void h4_issue_mmas(uint32_t d_tmem, uint32_t plane1_addr, uint32_t plane2_addr, uint32_t bank_addr, int ks,
                                              int pad_bytes, int tlo, int thi) {
  constexpr uint32_t kBankRows = PAIR ? 96 : 128;
  const uint64_t da1 = umma_desc_sw128(plane1_addr), da2 = umma_desc_sw128(plane2_addr);
  const uint64_t db = ptx::umma_desc(bank_addr, kBankRows * 16, 128);                          // N = 128 operand: bank rows from 0
  const uint64_t db64 = PAIR ? ptx::umma_desc(bank_addr + 64 * 16, kBankRows * 16, 128) : db;  // N = 64 operand
  constexpr uint32_t m = PAIR ? 256 : 128;
  constexpr uint32_t idesc128 = ptx::umma_idesc_f16(m, 128), idesc64 = ptx::umma_idesc_f16(m, 64);
  constexpr uint32_t kStep = 2 * kBankRows;  // descriptor units (16 B) per K-step of the bank
  auto a_step = [&](int s) {                 // K-step s starts 32 s (+ pad) bytes into row i: 128-byte rows, 16-byte descriptor units
    const uint32_t byte = 32u * (uint32_t)s + (uint32_t)pad_bytes;
    return (uint64_t)(8u * (byte >> 7) + ((byte >> 4) & 7u));
  };
  auto mma = [&](uint32_t d, uint64_t a, uint64_t bdesc, uint32_t idesc, bool acc) {
    if constexpr (PAIR) ptx::umma_pair_f16(d, a, bdesc, idesc, acc);
    else ptx::umma_f16(d, a, bdesc, idesc, acc);
  };
  for (int s = tlo; s < ks - thi; ++s) mma(d_tmem, da1 + a_step(s), db + (uint64_t)(kStep * s), idesc128, s != tlo);  // initialises all 128 columns
  for (int s = 0; s < tlo; ++s) mma(d_tmem, da1 + a_step(s), db64 + (uint64_t)(kStep * s), idesc64, true);
  for (int s = ks - thi; s < ks; ++s) mma(d_tmem, da1 + a_step(s), db64 + (uint64_t)(kStep * s), idesc64, true);
  for (int s = tlo; s < ks - thi; ++s) mma(d_tmem + 64u, da2 + a_step(s), db64 + (uint64_t)(kStep * s), idesc64, true);  // second-term columns
}

// two-term fp16 split of a pair with the residual scaled into the normal range: v = h1 + 2^-11 h2' (exact residual, |h2'| <= |v|)
__device__ __forceinline__ void split2_f16s(float a, float b, uint32_t& h1_bits, uint32_t& h2_bits) {
  const __half2 h1 = __floats2half2_rn(a, b);
  const float2 h1f = __half22float2(h1);
  // (v - h1) 2^11 as one packed FMA on the pre-scaled value: both products are exact (powers of two) and so is their difference
  const float2 r = __ffma2_rn(h1f, make_float2(-kH4Res, -kH4Res), __fmul2_rn(make_float2(a, b), make_float2(kH4Res, kH4Res)));
  const __half2 h2 = __floats2half2_rn(r.x, r.y);
  h1_bits = *reinterpret_cast<const uint32_t*>(&h1);
  h2_bits = *reinterpret_cast<const uint32_t*>(&h2);
}
// accumulator columns -> values: 2^-10 (D0 + 2^-11 D1), two adjacent columns at a time as packed FP32 (one FFMA2 + one FMUL2;
// per element an fma and a multiplication by a power of two)
__device__ __forceinline__ float2 h4_combine2(uint32_t d0a, uint32_t d0b, uint32_t d1a, uint32_t d1b) {
  const float2 t = __ffma2_rn(make_float2(__uint_as_float(d1a), __uint_as_float(d1b)), make_float2(1.0f / kH4Res, 1.0f / kH4Res),
                              make_float2(__uint_as_float(d0a), __uint_as_float(d0b)));
  constexpr float kInv = 1.0f / (float)(1 << kH16ScaleLog2);
  return __fmul2_rn(t, make_float2(kInv, kInv));
}

template <int N>
__device__ __forceinline__ void h4_tmem_ld(uint32_t taddr, uint32_t (&r)[N]) {
  static_assert(N == 2 || N == 4 || N == 8 || N == 16 || N == 32, "columns per load");
  if constexpr (N == 2) ptx::tmem_ld2(taddr, r);
  else if constexpr (N == 4) ptx::tmem_ld4(taddr, r);
  else if constexpr (N == 8) ptx::tmem_ld8(taddr, r);
  else if constexpr (N == 16) ptx::tmem_ld16(taddr, r);
  else ptx::tmem_ld32(taddr, r);
}

// eight samples -> their two fp16 terms: one 16-byte chunk at (swizzled) byte `off` of each plane of a pair, the second plane `plane` bytes
// after the first
__device__ __forceinline__ void h4_split_store8(const float (&w)[8], unsigned char* p1, int plane, uint32_t off) {
  uint4 a, bq;
  split2_f16s(w[0], w[1], a.x, bq.x);
  split2_f16s(w[2], w[3], a.y, bq.y);
  split2_f16s(w[4], w[5], a.z, bq.z);
  split2_f16s(w[6], w[7], a.w, bq.w);
  unsigned char* p2 = p1 + plane;
  *reinterpret_cast<uint4*>(p1 + off) = a;
  *reinterpret_cast<uint4*>(p2 + off) = bq;
}

// synthesis convert, n_band >= 8: v[kk] = four frames of band 8 bg + kk; chunk j = frame j of them, odd bands sign-flipped by fl
__device__ __forceinline__ void h4_synthesis_chunk8(const float4 (&v)[8], int j, uint32_t fl, float (&w)[8]) {
#pragma unroll
  for (int kk = 0; kk < 8; ++kk) {
    const float t = j == 0 ? v[kk].x : j == 1 ? v[kk].y : j == 2 ? v[kk].z : v[kk].w;
    w[kk] = (kk & 1) ? __uint_as_float(__float_as_uint(t) ^ fl) : t;
  }
}

// analysis drain, D (TMEM) -> v: worker thread (row i = tid & 127, band half hb = tid >> 7) gets frames FR i .. FR i + FR - 1 of bands
// HB hb .. HB hb + HB - 1 with the sign applied.  sigma(k, n): odd bands flip on even frames.  A row's first frame is a multiple of FR,
// even for FR > 1, so there the frame parity is dl's; `first` is the parity of the row's first frame, used at FR = 1 only.
template <int M>
__device__ __forceinline__ void h4_drain_analysis(uint32_t tmem, int dbuf, int tid, int first, int parity, float (&v)[64 / M][M / 2]) {
  constexpr int FR = 64 / M, HB = M / 2;
  const uint32_t taddr = tmem + ((uint32_t)(((tid >> 5) & 3) * 32) << 16) + (uint32_t)(dbuf * 128 + HB * (tid >> 7));
  uint32_t r0[FR][HB], r1[FR][HB];
#pragma unroll
  for (int dl = 0; dl < FR; ++dl) {
    h4_tmem_ld<HB>(taddr + dl * M, r0[dl]);
    h4_tmem_ld<HB>(taddr + 64 + dl * M, r1[dl]);
  }
  ptx::tmem_ld_wait();
#pragma unroll
  for (int dl = 0; dl < FR; ++dl) {
    const uint32_t flip = (((FR > 1 ? dl : first) + parity) & 1) == 0 ? 0x80000000u : 0u;
#pragma unroll
    for (int kk = 0; kk < HB; kk += 2) {
      const float2 t = h4_combine2(r0[dl][kk], r0[dl][kk + 1], r1[dl][kk], r1[dl][kk + 1]);
      v[dl][kk] = t.x;
      v[dl][kk + 1] = __uint_as_float(__float_as_uint(t.y) ^ flip);
    }
  }
}

// synthesis drain, D (TMEM) -> val.  Worker thread (row i, half hb) reads 32 consecutive output samples = four 32-byte chunks, but rows
// are 256 B apart: stored like that, every warp store would touch 32 lines.  A 4 x 4 chunk transpose inside each lane quad (two shuffle
// stages) leaves lane r with chunk r & 3 of the quad's four rows: val[q] = samples 32 hb + 8 (lane & 3) .. + 7 of row (i & ~3) | q, so
// one STG.256 per slot covers eight whole 128-byte lines.
__device__ __forceinline__ void h4_drain_synthesis(uint32_t tmem, int dbuf, int tid, float (&val)[4][8]) {
  const int hb = tid >> 7, lane = tid & 31;
  const uint32_t taddr = tmem + ((uint32_t)(((tid >> 5) & 3) * 32) << 16) + (uint32_t)(dbuf * 128 + 2 * hb * 16);
  uint32_t r0[2][16], r1[2][16];
  ptx::tmem_ld16(taddr, r0[0]);
  ptx::tmem_ld16(taddr + 64, r1[0]);
  ptx::tmem_ld16(taddr + 16, r0[1]);
  ptx::tmem_ld16(taddr + 80, r1[1]);
  ptx::tmem_ld_wait();
#pragma unroll
  for (int q = 0; q < 4; ++q)  // chunk q = samples 32 hb + 8 q .. + 7 of the row
#pragma unroll
    for (int e = 0; e < 8; e += 2) {
      const int c0 = 8 * (q & 1) + e;
      const float2 t = h4_combine2(r0[q >> 1][c0], r0[q >> 1][c0 + 1], r1[q >> 1][c0], r1[q >> 1][c0 + 1]);
      val[q][e] = t.x;
      val[q][e + 1] = t.y;
    }
  const bool b0 = lane & 1, b1 = lane & 2;
#pragma unroll
  for (int pr = 0; pr < 2; ++pr)  // lanes r, r ^ 1 swap the off-diagonal chunks of (2 pr, 2 pr + 1)
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float recv = __shfl_xor_sync(0xffffffffu, b0 ? val[2 * pr][e] : val[2 * pr + 1][e], 1);
      val[2 * pr + 1][e] = b0 ? val[2 * pr + 1][e] : recv;
      val[2 * pr][e] = b0 ? recv : val[2 * pr][e];
    }
#pragma unroll
  for (int u = 0; u < 2; ++u)  // lanes r, r ^ 2 swap the off-diagonal chunks of (u, u + 2)
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float recv = __shfl_xor_sync(0xffffffffu, b1 ? val[u][e] : val[u + 2][e], 2);
      val[u + 2][e] = b1 ? val[u + 2][e] : recv;
      val[u][e] = b1 ? recv : val[u][e];
    }
}

// PQMF_H4_TRACE (experiments/trace_h4.cu): `trace` = [iterations][8 warps][8] clock64 stamps of CTA 0 at the phase boundaries of the
// worker loop, then per CTA its lifetime in cycles and ns.  Kernels without a trace buffer pass nullptr.
#ifdef PQMF_H4_TRACE
#define H4_TRACE_PARAM , long long* trace
#define H4_TRACE(x) , x
#define H4_STAMP(k) do { if (trace && blockIdx.x == 0 && (tid & 31) == 0 && it < 64) trace[((size_t)it * 8 + (tid >> 5)) * 8 + (k)] = clock64(); } while (0)
#else
#define H4_TRACE_PARAM
#define H4_TRACE(x)
#define H4_STAMP(k) do { } while (0)
#endif

// shared-memory carve-up common to all Hankel-4 kernels
struct H4Smem {
  unsigned char *bank, *planes;
  uint64_t *pfull, *mma_bar, *bankfull;
  uint32_t* tmem_slot;
};
__device__ __forceinline__ H4Smem h4_carve(unsigned char* smem, const H4Shape& g) {
  H4Smem s;
  s.bank = smem;
  s.planes = smem + g.bank;
  s.pfull = reinterpret_cast<uint64_t*>(smem + g.bank + 4 * g.plane);  // [2]
  s.mma_bar = s.pfull + 2;                                              // [2]
  s.bankfull = s.mma_bar + 2;
  s.tmem_slot = reinterpret_cast<uint32_t*>(s.bankfull + 1);
  return s;
}

// barrier init, TMEM allocation, bank staging.  pfull lives in the leader CTA (rank 0): one arrival per worker warp of every
// CTA of the pair.  Returns the TMEM base address.
template <bool PAIR>
__device__ __forceinline__ uint32_t h4_prologue(const H4Smem& s, const H4Shape& g, const uint16_t* bank_images, uint32_t rank, int worker_warps,
                                                int tid) {
  const int warp = tid >> 5;
  ptx::grid_dep_launch();  // the next kernel in the stream may set itself up while this one is still running
  if (tid == 0) {
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&s.pfull[i], worker_warps * (PAIR ? 2 : 1));
      ptx::mbar_init(&s.mma_bar[i], 1);
    }
    ptx::mbar_init(s.bankfull, 1);
    ptx::fence_barrier_init();
    // the bank image streams in while the TMEM allocation and the barriers below complete
    ptx::mbar_arrive_expect_tx(s.bankfull, (uint32_t)g.bank);
    ptx::bulk_g2s(s.bank, reinterpret_cast<const unsigned char*>(bank_images) + (size_t)rank * g.bank, (uint32_t)g.bank, s.bankfull);
  }
  if (warp == 0) {
    if constexpr (PAIR) {
      ptx::tmem_alloc_pair(s.tmem_slot, 256);
    } else {
      ptx::tmem_alloc(s.tmem_slot, 256);
      ptx::tmem_relinquish();
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if constexpr (PAIR) ptx::cluster_sync_all();  // the peer's barriers are initialised before anyone arrives on them
  ptx::tc_fence_after();
  ptx::grid_dep_wait();  // everything above overlapped the previous kernel's tail; its results (and its reads of our outputs) are done now
  return *s.tmem_slot;
}

template <bool PAIR>
__device__ __forceinline__ void h4_teardown(uint32_t tmem, int warp) {
  ptx::tc_fence_before();
  __syncthreads();
  if constexpr (PAIR) {
    ptx::cluster_sync_all();  // the peer may still be read by / signalled from the leader's last MMAs
    if (warp == 0) ptx::tmem_dealloc_pair(tmem, 256);
  } else {
    if (warp == 0) ptx::tmem_dealloc(tmem, 256);
  }
}

// the issuer warp's loop (leader CTA only): tcgen05.mma issue blocks once the tensor pipe's queue is full (a 54-MMA group keeps
// the issuing thread for ~3200 cycles), so this warp does nothing else and the pipe never waits for a converting thread
template <bool PAIR>
__device__ __forceinline__ void h4_issuer_loop(const H4Smem& s, const H4Shape& g, uint32_t tmem, unsigned n_iter, int pad_bytes, int tlo,
                                               int thi) {
  const uint32_t bank_addr = ptx::smem_u32(s.bank), plane_addr = ptx::smem_u32(s.planes);
  for (unsigned it = 0; it < n_iter; ++it) {
    const int pb = (int)(it & 1);
    ptx::mbar_wait(&s.pfull[pb], (it >> 1) & 1);
    ptx::tc_fence_after();
    if (ptx::elect_one_sync()) {
      h4_issue_mmas<PAIR>(tmem + (uint32_t)(pb * 128), plane_addr + (2 * pb) * g.plane, plane_addr + (2 * pb + 1) * g.plane, bank_addr, g.ks,
                          pad_bytes, tlo, thi);
      if constexpr (PAIR) ptx::umma_pair_commit(&s.mma_bar[pb]);
      else ptx::umma_commit(&s.mma_bar[pb]);
    }
    __syncwarp();
  }
}

// a worker warp publishes its share of planes[pb]: one arrival per warp, after this CTA's bank image has landed (the first tile waits
// for it)
template <bool PAIR>
__device__ __forceinline__ void h4_publish(const H4Smem& s, uint32_t pfull_leader, unsigned it, int pb, int tid) {
  ptx::fence_proxy_async();
  ptx::tc_fence_before();
  __syncwarp();
  if ((tid & 31) == 0) {
    if (it == 0) ptx::mbar_wait(s.bankfull, 0);
    if constexpr (PAIR) ptx::mbar_arrive_cluster(pfull_leader + 8u * pb);
    else ptx::mbar_arrive(&s.pfull[pb]);
  }
}

// the worker warps' tile loop.  Iteration it converts tile it into planes[it & 1] and publishes it, loads tile it + 1 into registers
// (one tile ahead), then waits for the MMAs of tile it - 1 -- after which planes[(it - 1) & 1] may be rewritten -- and drains their
// accumulator.  The kernel supplies the steps: convert(pb) the current tile, load_next() the tile after it, drain(dbuf) the previous
// tile, advance() the cursors (current -> previous, next -> current).
template <bool PAIR, typename Convert, typename LoadNext, typename Drain, typename Advance>
__device__ __forceinline__ void h4_worker_loop(const H4Smem& s, uint32_t pfull_leader, unsigned n_iter, int tid, Convert&& convert,
                                               LoadNext&& load_next, Drain&& drain, Advance&& advance H4_TRACE_PARAM) {
  for (unsigned it = 0; it < n_iter; ++it) {
    const int pb = (int)(it & 1);
    H4_STAMP(0);
    convert(pb);
    H4_STAMP(1);
    h4_publish<PAIR>(s, pfull_leader, it, pb, tid);
    if (it + 1 < n_iter) load_next();  // consumed at the top of the next iteration
    H4_STAMP(2);
    if (it > 0) {
      ptx::mbar_wait(&s.mma_bar[(it - 1) & 1], ((it - 1) >> 1) & 1);
      ptx::tc_fence_after();
      drain((int)((it - 1) & 1));
    }
    H4_STAMP(5);
    advance();
  }
  ptx::mbar_wait(&s.mma_bar[(n_iter - 1) & 1], ((n_iter - 1) >> 1) & 1);
  ptx::tc_fence_after();
  drain((int)((n_iter - 1) & 1));
}

// the frame of every Hankel-4 kernel: shared-memory carve-up, prologue, the issuer warp (warp WORKERS / 32, leader CTA only) and the
// teardown.  Each CTA (pair) runs visits x its share of the n_tiles tiles; the worker warps run
// workers(smem, tmem, pfull_leader, n_iter).
template <bool PAIR, int WORKERS, typename Workers>
__device__ __forceinline__ void h4_kernel(const H4Shape& g, const uint16_t* bank, long n_tiles, unsigned visits, int pad_bytes, int trim_lo,
                                          int trim_hi, Workers&& workers H4_TRACE_PARAM) {
  extern __shared__ __align__(1024) unsigned char h4_smem[];
  const H4Smem sm = h4_carve(h4_smem, g);
  const int tid = threadIdx.x, warp = tid >> 5;
  const uint32_t rank = PAIR ? ptx::cluster_ctarank() : 0u;
  const uint32_t tmem = h4_prologue<PAIR>(sm, g, bank, rank, WORKERS / 32, tid);
  const uint32_t pfull_leader = PAIR ? ptx::mapa_shared(ptx::smem_u32(sm.pfull), 0) : 0u;
  const unsigned first_tile = PAIR ? (blockIdx.x & ~1u) : blockIdx.x;  // both CTAs of a pair run the same number of tiles
  const unsigned n_iter = visits * (unsigned)((n_tiles - first_tile + gridDim.x - 1) / gridDim.x);
#ifdef PQMF_H4_TRACE
  long long cta_c0 = clock64(), cta_t0;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(cta_t0));
#endif
  if (warp == WORKERS / 32) {
    if (rank == 0) h4_issuer_loop<PAIR>(sm, g, tmem, n_iter, pad_bytes, trim_lo, trim_hi);
  } else {
    workers(sm, tmem, pfull_leader, n_iter);
  }
#ifdef PQMF_H4_TRACE
  __syncthreads();
  if (trace && tid == 0) {
    long long t1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
    trace[64 * 64 + 2 * blockIdx.x] = clock64() - cta_c0;
    trace[64 * 64 + 2 * blockIdx.x + 1] = t1 - cta_t0;
  }
#endif
  h4_teardown<PAIR>(tmem, warp);
}

// =============================================================================================
// analysis
// =============================================================================================
struct H4AnalysisParams {
  const float* x;        // [B, T]; half-precision instantiations: raw fp16 / bf16 bits (the launch's H4Io)
  PcmIn in;              // PCM instantiation: the rows come from interleaved int16 WAV frames (x unused)
  float* y;              // [B, M, F]; half-precision instantiations: raw fp16 / bf16 bits
  const uint16_t* bank;  // fp16 image(s), see hankel4_build_banks / hankel4_pair_image
  long T, F;
  int off;               // L / 2 (offline only: streaming blocks are far smaller than a tile)
  int parity;
  int trim_lo, trim_hi;  // edge K-steps without correction terms (h4_issue_mmas)
  int accumulate;        // add to what y already holds (second launch of a bank split in two tap ranges)
  int keep_in_l2;        // store y without the streaming hint: a synthesis launch that follows walks the tiles backwards and finds the tail in L2
  H4Shape g;
  long tiles_per_row, n_tiles;
#ifdef PQMF_H4_TRACE
  long long* trace;      // [iterations][8 warps][8] clock64 stamps of CTA 0 (experiments/trace_h4.cu)
#endif
};

template <int M, bool PAIR, H4Io IO>
__global__ void __launch_bounds__(kH4Threads, 1) h4_analysis_kernel(H4AnalysisParams p) {
  h4_kernel<PAIR, kH4Workers>(p.g, p.bank, p.n_tiles, 1u, 0, p.trim_lo, p.trim_hi, [&](const H4Smem& sm, uint32_t tmem, uint32_t pfull_leader, unsigned n_iter) {
    constexpr bool PCM = IO == H4Io::PCM, HALF = h4_io_half(IO);
    constexpr int FR = 64 / M;                                               // frames per 64-sample row
    constexpr int HB = M / 2;                                                // bands per epilogue thread
    constexpr int NO = (kH4MaxPlaneRows * 8 + kH4Workers - 1) / kH4Workers;  // 8-sample loads per thread per tile (a row is 8 of them)
    const H4Shape& g = p.g;
    const int tid = threadIdx.x;
    const unsigned tpr = (unsigned)p.tiles_per_row;
    const unsigned step_b = gridDim.x / tpr, step_c = gridDim.x % tpr;
    const unsigned n_rows = (unsigned)(p.n_tiles / p.tiles_per_row);  // a tile with b >= n_rows is padding (zeros in, nothing out)
    auto advance = [&](unsigned& bb, unsigned& cc) {
      bb += step_b;
      cc += step_c;
      if (cc >= tpr) {
        cc -= tpr;
        ++bb;
      }
    };
    unsigned b = blockIdx.x / tpr, c = blockIdx.x % tpr;  // tile it
    unsigned b1 = b, c1 = c;                              // tile it + 1
    advance(b1, c1);
    unsigned prev_b = 0, prev_c = 0;                      // tile it - 1
    const int n_octs = g.rows * 8;
    // this thread's share of the fp32 window of a tile (8 consecutive samples per 256-bit load), prefetched one tile ahead straight
    // from global memory.  (Two tiles ahead in two register sets was measured on the same box: 6 % slower in bursts and sustained --
    // the extra live registers cost more than the latency they hide.)
    float x0[NO][8];
    auto load_window = [&](unsigned bb, unsigned cc) {
      const long s0 = (long)cc * kH4TileSamples + g.jlo - p.off;
      const float* xrow = p.x + (size_t)bb * p.T;
      const uint16_t* xhrow = reinterpret_cast<const uint16_t*>(p.x) + (size_t)bb * p.T;
#pragma unroll
      for (int r = 0; r < NO; ++r) {
        const int o = tid + kH4Workers * r;
        const long s = s0 + 8L * o;
        if (bb < n_rows && o < n_octs && s >= 0 && s < p.T) {
          if constexpr (PCM) {
            pcm_load8_raw(p.in, bb, s, p.T, x0[r]);   // raw int16 words: converted when the tile is consumed
          } else if constexpr (HALF) {                // eight half samples = 16 bytes, kept raw in x0[r][0..3] until the tile is consumed
            const float4 raw = ptx::ldg128_na(reinterpret_cast<const float4*>(xhrow + s));
            x0[r][0] = raw.x; x0[r][1] = raw.y; x0[r][2] = raw.z; x0[r][3] = raw.w;
          } else {
            ptx::ldg256_na(xrow + s, x0[r]);
          }
        } else {
#pragma unroll
          for (int e = 0; e < 8; ++e) x0[r][e] = 0.f;
        }
      }
    };
    // fp32 window -> two fp16 planes (SWIZZLE_128B rows of 64 samples, one 16-byte chunk per load).  planes[pb] were last read by
    // the MMAs of tile it-2, whose completion this thread observed before draining tile it-2.
    auto convert = [&](int pb) {
      unsigned char* p1 = sm.planes + (2 * pb) * g.plane;
#pragma unroll
      for (int r = 0; r < NO; ++r) {
        const int o = tid + kH4Workers * r;
        if (o < n_octs) {
          if constexpr (PCM) {  // the registers hold raw PCM words where the load was live (zeros stay zeros: 0 is not a valid raw mono / stereo pattern to convert)
            const long s = (long)c * kH4TileSamples + g.jlo - p.off + 8L * o;
            if (b < n_rows && s >= 0 && s < p.T) pcm_convert8(p.in, b, x0[r]);
          }
          if constexpr (HALF) h4_widen8<IO>(x0[r]);  // exact; zero words (padding) widen to zeros
          h4_split_store8(x0[r], p1, g.plane, sw128_offset((uint32_t)o * 16u));
        }
      }
    };
    // D (TMEM) -> y: thread (row i, band half hb) owns frames FR i .. FR i + FR - 1 of bands HB hb .. HB hb + HB - 1:
    // FR consecutive frames per band (32 / 16 / 8 bytes at n_band 8 / 16 / 32), consecutive rows in consecutive lanes
    auto drain = [&](int dbuf) {
      if (prev_b >= n_rows) return;
      const int i = tid & 127, hb = tid >> 7;
      const long n = ((long)prev_c * kH4Rows + i) * FR;
      float v[FR][HB];
      h4_drain_analysis<M>(tmem, dbuf, tid, (int)(n & 1), p.parity, v);
      if constexpr (HALF) {  // round to nearest even; FR consecutive frames = 2 FR bytes per band (no accumulation: split banks are not native)
        uint16_t* yp = reinterpret_cast<uint16_t*>(p.y) + ((size_t)prev_b * M + HB * hb) * p.F + n;
        if (n + FR - 1 < p.F && (p.F % (FR >= 8 ? 8 : FR)) == 0) {
#pragma unroll
          for (int kk = 0; kk < HB; ++kk) {
            uint16_t* q = yp + (size_t)kk * p.F;
            if constexpr (FR >= 8) {
#pragma unroll
              for (int d8 = 0; d8 < FR; d8 += 8) {
                const uint4 w = make_uint4(h4_narrow2<IO>(v[d8][kk], v[d8 + 1][kk]), h4_narrow2<IO>(v[d8 + 2][kk], v[d8 + 3][kk]),
                                           h4_narrow2<IO>(v[d8 + 4][kk], v[d8 + 5][kk]), h4_narrow2<IO>(v[d8 + 6][kk], v[d8 + 7][kk]));
                if (p.keep_in_l2) *reinterpret_cast<uint4*>(q + d8) = w;
                else __stcs(reinterpret_cast<uint4*>(q + d8), w);
              }
            } else if constexpr (FR == 4) {
              const uint2 w = make_uint2(h4_narrow2<IO>(v[0][kk], v[1][kk]), h4_narrow2<IO>(v[2][kk], v[3][kk]));
              if (p.keep_in_l2) *reinterpret_cast<uint2*>(q) = w;
              else __stcs(reinterpret_cast<uint2*>(q), w);
            } else if constexpr (FR == 2) {
              __stcs(reinterpret_cast<unsigned int*>(q), h4_narrow2<IO>(v[0][kk], v[1][kk]));
            } else {
              __stcs(reinterpret_cast<unsigned short*>(q), h4_narrow1<IO>(v[0][kk]));
            }
          }
        } else {
#pragma unroll
          for (int kk = 0; kk < HB; ++kk)
#pragma unroll
            for (int dl = 0; dl < FR; ++dl)
              if (n + dl < p.F) yp[(size_t)kk * p.F + dl] = h4_narrow1<IO>(v[dl][kk]);
        }
        return;
      }
      float* yp = p.y + ((size_t)prev_b * M + HB * hb) * p.F + n;
      if (n + FR - 1 < p.F && (p.F % (FR >= 4 ? 4 : FR)) == 0) {
        if (p.accumulate) {  // second tap range of a split bank: all the reads first, so they overlap instead of alternating with the stores
          float prev[FR][HB];
#pragma unroll
          for (int kk = 0; kk < HB; ++kk)
#pragma unroll
            for (int dl = 0; dl < FR; ++dl) prev[dl][kk] = __ldcs(yp + (size_t)kk * p.F + dl);
#pragma unroll
          for (int kk = 0; kk < HB; ++kk)
#pragma unroll
            for (int dl = 0; dl < FR; ++dl) v[dl][kk] += prev[dl][kk];
        }
#pragma unroll
        for (int kk = 0; kk < HB; ++kk) {
          float* q = yp + (size_t)kk * p.F;
          if constexpr (FR >= 4) {
#pragma unroll
            for (int d4 = 0; d4 < FR; d4 += 4) {
              const float4 w = make_float4(v[d4][kk], v[d4 + 1][kk], v[d4 + 2][kk], v[d4 + 3][kk]);
              if (p.keep_in_l2) *reinterpret_cast<float4*>(q + d4) = w;
              else __stcs(reinterpret_cast<float4*>(q + d4), w);
            }
          } else if constexpr (FR == 2) {
            __stcs(reinterpret_cast<float2*>(q), make_float2(v[0][kk], v[1][kk]));
          } else {
            __stcs(q, v[0][kk]);
          }
        }
      } else {
#pragma unroll
        for (int kk = 0; kk < HB; ++kk)
#pragma unroll
          for (int dl = 0; dl < FR; ++dl)
            if (n + dl < p.F) yp[(size_t)kk * p.F + dl] = v[dl][kk] + (p.accumulate ? yp[(size_t)kk * p.F + dl] : 0.f);
      }
    };

    load_window(b, c);
    h4_worker_loop<PAIR>(sm, pfull_leader, n_iter, tid, convert, [&] { load_window(b1, c1); }, drain, [&] {
      prev_b = b;
      prev_c = c;
      b = b1;
      c = c1;
      advance(b1, c1);
    } H4_TRACE(p.trace));
  } H4_TRACE(p.trace));
}

// =============================================================================================
// synthesis
// =============================================================================================
struct H4SynthesisParams {
  const float* s;        // [B, M, F]; half-precision instantiations: raw fp16 / bf16 bits (the launch's H4Io)
  float* out;            // [B, M F]; half-precision instantiations: raw fp16 / bf16 bits
  int16_t* pcm_out;      // PCM instantiation: interleaved int16 WAV frames [B / C, M F, C] (out unused)
  int C;
  int duo;               // PCM stereo: the launch walks CLIPS; a CTA runs the left and the right row of a tile back to back and its
                         // epilogue threads -- which hold the same eight samples of both -- store whole interleaved 32-byte groups
  const uint16_t* bank;
  long F;
  int o;                 // off2 / M: L / (2 M) (PQMF.inverse) or one less (CachedPQMF.inverse)
  int parity;
  int trim_lo, trim_hi;
  int accumulate;        // add to what out already holds
  int reverse;           // walk the tiles from the last to the first (see H4AnalysisParams::keep_in_l2)
  H4Shape g;
  long tiles_per_row, n_tiles;
#ifdef PQMF_H4_TRACE
  long long* trace;
#endif
};

template <int M, bool PAIR, H4Io IO>
__global__ void __launch_bounds__(kH4SynThreads, 1) h4_synthesis_kernel(H4SynthesisParams p) {
  constexpr bool PCM = IO == H4Io::PCM, HALF = h4_io_half(IO);
  // plane frame m <-> sub-band frame n = 128 FR c + (o - ehi - pad) + m, ehi = largest frame lag with a non-zero tap,
  // pad = (o - ehi) mod 4, so that frame quads are 16-byte aligned in global memory; K-step s of row i then starts
  // 32 s + 2 M pad bytes into the row.
  const int ehi = (p.g.jlo + p.g.kt) / M - 1;
  const int pad = (p.o - ehi) & 3;
  const unsigned G = (PCM && p.duo) ? 2u : 1u;  // rows per tile visit (see H4SynthesisParams::duo): b counts clips then, row = G b + channel
  h4_kernel<PAIR, kH4SynWorkers>(p.g, p.bank, p.n_tiles, G, 2 * M * pad, p.trim_lo, p.trim_hi, [&](const H4Smem& sm, uint32_t tmem, uint32_t pfull_leader, unsigned n_iter) {
    constexpr int FR = 64 / M;                // frames per 128-byte plane row ([frame][band] fp16)
    constexpr int NBG = M >= 8 ? M / 8 : 1;   // band groups: a 16-byte chunk is 8 bands of one frame, or (n_band 4) all bands of two frames
    constexpr int FPI = M >= 8 ? 4 : 32 / M;  // frames per load/convert item (four chunks)
    const H4Shape& g = p.g;
    const int tid = threadIdx.x, warp = tid >> 5;
    const int nbase = p.o - ehi - pad;  // multiple of 4 (may be negative)
    const unsigned tpr = (unsigned)p.tiles_per_row;
    const unsigned step_b = gridDim.x / tpr, step_c = gridDim.x % tpr;
    const unsigned n_rows = (unsigned)(p.n_tiles / p.tiles_per_row);
    auto next_visit = [&](unsigned& bb, unsigned& cc, unsigned& hh) {  // the tile's next row, or the CTA's next tile
      if (++hh == G) {
        hh = 0;
        bb += step_b;
        cc += step_c;
        if (cc >= tpr) {
          cc -= tpr;
          ++bb;
        }
      }
    };
    unsigned b = blockIdx.x / tpr, c = blockIdx.x % tpr, h = 0;  // visit it
    unsigned b1 = b, c1 = c, h1 = 0;                             // visit it + 1
    next_visit(b1, c1, h1);
    unsigned prev_b = 0, prev_c = 0, prev_h = 0;                 // visit it - 1
    // ---- Item (fq, bg): frames 4 fq .. 4 fq + 3 of bands 8 bg .. 8 bg + 7 = eight float4 loads (prefetched one tile ahead) -> four
    //      16-byte chunks per fp16 plane.  bg-major thread order keeps a quarter-warp on eight consecutive frame quads of one band
    //      group: their SWIZZLE_128B images hit eight different bank groups at n_band 8 and 16.
    const int n_fq = (g.rows * FR + FPI - 1) / FPI;  // items per band group (the last one may run into the plane's padding)
    const int bg = tid / n_fq, fq = tid - bg * n_fq;
    const bool has_item = tid < n_fq * NBG;
    float4 v0[8];  // prefetched one tile ahead (half instantiations: four raw frames in .x / .y, widened when the tile is consumed)
    auto load4h = [&](const uint16_t* at, bool ok) {  // four half frames of one band
      if (!ok) return make_float4(0.f, 0.f, 0.f, 0.f);
      const float2 raw = ptx::ldg64_na(at);
      return make_float4(raw.x, raw.y, 0.f, 0.f);
    };
    auto load_frames = [&](unsigned bb, unsigned cc, unsigned hh) {
      if (p.reverse && bb < n_rows) {
        bb = n_rows - 1 - bb;
        cc = tpr - 1 - cc;
      }
      const long n = (long)cc * (kH4Rows * FR) + nbase + FPI * fq;
      const bool live = bb < n_rows && has_item;
      const size_t row = (size_t)bb * G + hh;
      if constexpr (HALF) {    // the same frames as below, 8 bytes per load
        if constexpr (M >= 8) {
          const uint16_t* sp = reinterpret_cast<const uint16_t*>(p.s) + (row * M + 8 * bg) * p.F + n;
          const bool ok = live && n >= 0 && n + 3 < p.F;
#pragma unroll
          for (int kk = 0; kk < 8; ++kk) v0[kk] = load4h(sp + (size_t)kk * p.F, ok);
        } else {
          const uint16_t* sp = reinterpret_cast<const uint16_t*>(p.s) + row * M * p.F + n;
#pragma unroll
          for (int kk = 0; kk < 8; ++kk) {
            const int b4 = kk >> 1, hf = kk & 1;
            v0[kk] = load4h(sp + (size_t)b4 * p.F + 4 * hf, live && n + 4 * hf >= 0 && n + 4 * hf + 3 < p.F);
          }
        }
      } else if constexpr (M >= 8) {  // v0[kk] = frames n .. n + 3 of band 8 bg + kk
        const float* sp = p.s + (row * M + 8 * bg) * p.F + n;
        const bool ok = live && n >= 0 && n + 3 < p.F;
#pragma unroll
        for (int kk = 0; kk < 8; ++kk) v0[kk] = ok ? ptx::ldg128_na(reinterpret_cast<const float4*>(sp + (size_t)kk * p.F)) : make_float4(0.f, 0.f, 0.f, 0.f);
      } else {                 // n_band 4: v0[2 b + h] = frames n + 4 h .. n + 4 h + 3 of band b
        const float* sp = p.s + row * M * p.F + n;
#pragma unroll
        for (int kk = 0; kk < 8; ++kk) {
          const int b4 = kk >> 1, hf = kk & 1;
          const bool ok = live && n + 4 * hf >= 0 && n + 4 * hf + 3 < p.F;
          v0[kk] = ok ? ptx::ldg128_na(reinterpret_cast<const float4*>(sp + (size_t)b4 * p.F + 4 * hf)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
    };
    // sigma(k, n): odd bands (odd kk) flip on even global frames; quads start on multiples of 4, so the parity is j's
    const uint32_t flip_even = (p.parity & 1) ? 0u : 0x80000000u, flip_odd = flip_even ^ 0x80000000u;
    auto convert = [&](int pb) {
      float4 v[8];  // the tile's frames as fp32
#pragma unroll
      for (int kk = 0; kk < 8; ++kk) v[kk] = HALF ? h4_widen4<IO>(v0[kk]) : v0[kk];  // exact
      if (!has_item) return;
      unsigned char* p1 = sm.planes + (2 * pb) * g.plane;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float w[8];
        uint32_t o;
        if constexpr (M >= 8) {  // chunk j = frame 4 fq + j, bands 8 bg .. 8 bg + 7
          h4_synthesis_chunk8(v, j, (j & 1) ? flip_odd : flip_even, w);
          o = sw128_offset((uint32_t)(4 * fq + j) * (2u * M) + 16u * bg);
        } else {                 // n_band 4: chunk j = frames 8 fq + 2 j (even) and + 1 (odd), four bands each
#pragma unroll
          for (int kk = 0; kk < 8; ++kk) {
            const int b4 = kk & 3, odd = kk >> 2;
            const float4& q = v[2 * b4 + (j >> 1)];
            const int cmp = 2 * (j & 1) + odd;
            const float t = cmp == 0 ? q.x : cmp == 1 ? q.y : cmp == 2 ? q.z : q.w;
            w[kk] = (b4 & 1) ? __uint_as_float(__float_as_uint(t) ^ (odd ? flip_odd : flip_even)) : t;
          }
          o = sw128_offset((uint32_t)(8 * fq + 2 * j) * (2u * M));
        }
        h4_split_store8(w, p1, g.plane, o);
      }
    };
    // D (TMEM) -> out: h4_drain_synthesis leaves slot q with 8 samples of row (i & ~3) | q; one 32-byte store each
    uint32_t held[4][4];  // duo: the left channel's quantised samples of this thread's four chunks, kept for the right channel's visit
    auto drain = [&](int dbuf) {
      if (warp >= 8 || prev_b >= n_rows) return;  // every worker waited for the MMAs; the ninth warp has no TMEM rows to drain
      unsigned bb = prev_b, cc = prev_c;
      if (p.reverse) {
        bb = n_rows - 1 - bb;
        cc = tpr - 1 - cc;
      }
      const size_t row = (size_t)bb * G + prev_h;
      const int i = tid & 127, hb = tid >> 7, lane = tid & 31;
      float val[4][8];
      h4_drain_synthesis(tmem, dbuf, tid, val);
      // slot q holds samples 64 row + 32 hb + 8 (lane & 3) .. + 7 of the tile, row = (i & ~3) | q
      const long total = p.F * M;  // samples per output row (a multiple of 8: the dispatcher requires F % 4 == 0)
      const long t0 = (long)cc * kH4TileSamples + 64 * (i & ~3) + 32 * hb + 8 * (lane & 3);
      if constexpr (PCM) {
        if (G == 2) {
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            uint32_t w[4];
#pragma unroll
            for (int k = 0; k < 4; ++k)
              w[k] = (uint32_t)(uint16_t)pcm_quantise(val[q][2 * k]) | ((uint32_t)(uint16_t)pcm_quantise(val[q][2 * k + 1]) << 16);
            if (prev_h == 0) {
#pragma unroll
              for (int k = 0; k < 4; ++k) held[q][k] = w[k];
            } else if (t0 + 64 * q + 7 < total) {
              float lr[8];  // eight WAV frames (left | right << 16) as raw words
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                lr[2 * k] = __uint_as_float(__byte_perm(held[q][k], w[k], 0x5410));
                lr[2 * k + 1] = __uint_as_float(__byte_perm(held[q][k], w[k], 0x7632));
              }
              ptx::stg256_cs(reinterpret_cast<float*>(p.pcm_out + ((size_t)bb * total + t0 + 64 * q) * 2), lr);
            }
          }
          return;
        }
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (t0 + 64 * q + 7 < total) pcm_store8(p.pcm_out, p.C, (long)row, t0 + 64 * q, total, val[q]);
        return;
      }
      if constexpr (HALF) {  // round to nearest even: eight samples = one 16-byte store per slot, a lane quad covers 64 contiguous bytes
        uint16_t* op = reinterpret_cast<uint16_t*>(p.out) + row * total + t0;
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (t0 + 64 * q + 7 < total) {
            const uint4 w = make_uint4(h4_narrow2<IO>(val[q][0], val[q][1]), h4_narrow2<IO>(val[q][2], val[q][3]), h4_narrow2<IO>(val[q][4], val[q][5]),
                                       h4_narrow2<IO>(val[q][6], val[q][7]));
            __stcs(reinterpret_cast<uint4*>(op + (size_t)q * 64), w);
          }
        return;
      }
      float* op = p.out + row * total + t0;
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (t0 + 64 * q + 7 < total) {
          if (p.accumulate) {
            float prev[8];
            ptx::ldg256_cs(op + (size_t)q * 64, prev);
#pragma unroll
            for (int e = 0; e < 8; ++e) val[q][e] += prev[e];
          }
          ptx::stg256_cs(op + (size_t)q * 64, val[q]);
        }
    };

    load_frames(b, c, h);
    h4_worker_loop<PAIR>(sm, pfull_leader, n_iter, tid, convert, [&] { load_frames(b1, c1, h1); }, drain, [&] {
      prev_b = b;
      prev_c = c;
      prev_h = h;
      b = b1;
      c = c1;
      h = h1;
      next_visit(b1, c1, h1);
    } H4_TRACE(p.trace));
  } H4_TRACE(p.trace));
}

// ---------------------------------------------------------------------------------------------
// launches
// ---------------------------------------------------------------------------------------------
// per-kernel, per-device record of the dynamic shared memory opted into so far.  Several host threads may launch concurrently
// (one per device in pqmf_roundtrip_host_multi_f32): the values are atomics, and racing threads at worst both set the attribute.
struct H4Configured {
  std::atomic<int> bytes[64];
  H4Configured() {
    for (auto& b : bytes) b.store(0, std::memory_order_relaxed);
  }
};
inline int h4_sm_count(int dev) {
  static std::atomic<int> sm_count[64];
  int n = sm_count[dev].load(std::memory_order_relaxed);
  if (n == 0) {
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    n = n > 0 ? n : 148;
    sm_count[dev].store(n, std::memory_order_relaxed);
  }
  return n;
}
template <typename Kern>
inline int h4_configure(Kern kern, int bytes, H4Configured& configured, int& sm_count_out) {
  int dev = 0;
  cudaGetDevice(&dev);
  dev &= 63;
  if (configured.bytes[dev].load(std::memory_order_acquire) < bytes) {  // the opt-in limit only ever grows (shapes with more K-steps need more)
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e != cudaSuccess) return (int)e;
    int seen = configured.bytes[dev].load(std::memory_order_relaxed);
    while (seen < bytes && !configured.bytes[dev].compare_exchange_weak(seen, bytes, std::memory_order_release)) {
    }
  }
  sm_count_out = h4_sm_count(dev);
  return 0;
}

// the tiles of an offline launch: B rows of row_samples samples (analysis: input, synthesis: output); false: too many for the kernels'
// 32-bit tile cursors
template <typename Params>
inline bool h4_set_tiles(Params& p, int B, long row_samples) {
  p.tiles_per_row = (row_samples + kH4TileSamples - 1) / kH4TileSamples;
  p.n_tiles = p.tiles_per_row * B;
  return p.tiles_per_row < (1L << 31) && p.n_tiles < (1L << 40);
}

// one CTA (or CTA pair) per SM, static round-robin over the caller's p.n_tiles tiles; PAIR launches clusters of two
template <bool PAIR, typename Kern, typename Params>
inline int h4_launch(Kern kern, const Params& p, int threads, H4Configured& configured, cudaStream_t st) {
  int sms = 0;
  if (!h4_shape_fits(p.g)) return -2;
  if (int e = h4_configure(kern, p.g.bytes, configured, sms)) return e;
  long grid = PAIR ? (sms & ~1) : sms;
  const long want = PAIR ? ((p.n_tiles + 1) & ~1L) : p.n_tiles;
  if (grid > want) grid = want;
  if constexpr (PAIR) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3((unsigned)threads);
    cfg.dynamicSmemBytes = (size_t)p.g.bytes;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;  // start-up overlaps the previous kernel's tail (grid_dep_wait)
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 2;
    return (int)cudaLaunchKernelEx(&cfg, kern, p);
  } else {
    kern<<<(unsigned)grid, threads, p.g.bytes, st>>>(p);
    return (int)cudaGetLastError();
  }
}

// the PCM and half-precision instantiations exist as CTA pairs only (the single-CTA launch is a fallback for contexts that cannot
// co-schedule pairs)
template <int M, bool PAIR>
int h4_launch_analysis(H4AnalysisParams p, int B, cudaStream_t st, H4Io io = H4Io::F32) {
  static H4Configured configured[4];
  if (!h4_set_tiles(p, B, p.F * M)) return -2;
  if (io != H4Io::F32) {
    if constexpr (PAIR) {
      switch (io) {
        case H4Io::PCM: return h4_launch<PAIR>(h4_analysis_kernel<M, PAIR, H4Io::PCM>, p, kH4Threads, configured[1], st);
        case H4Io::F16: return h4_launch<PAIR>(h4_analysis_kernel<M, PAIR, H4Io::F16>, p, kH4Threads, configured[2], st);
        case H4Io::BF16: return h4_launch<PAIR>(h4_analysis_kernel<M, PAIR, H4Io::BF16>, p, kH4Threads, configured[3], st);
        default: return -2;
      }
    } else {
      return -2;
    }
  }
  return h4_launch<PAIR>(h4_analysis_kernel<M, PAIR, H4Io::F32>, p, kH4Threads, configured[0], st);
}

template <int M, bool PAIR>
int h4_launch_synthesis(H4SynthesisParams p, int B, cudaStream_t st, H4Io io = H4Io::F32) {
  static H4Configured configured[4];
  if (io == H4Io::PCM) {
    if constexpr (PAIR) {
      p.duo = (p.C == 2 && B % 2 == 0) ? 1 : 0;  // stereo: the tiles of a launch are (clip, chunk), each visited once per channel
      if (!h4_set_tiles(p, p.duo ? B / 2 : B, p.F * M)) return -2;
      return h4_launch<PAIR>(h4_synthesis_kernel<M, PAIR, H4Io::PCM>, p, kH4SynThreads, configured[1], st);
    } else {
      return -2;
    }
  }
  if (!h4_set_tiles(p, B, p.F * M)) return -2;
  if (h4_io_half(io)) {
    if constexpr (PAIR) {
      if (io == H4Io::F16) return h4_launch<PAIR>(h4_synthesis_kernel<M, PAIR, H4Io::F16>, p, kH4SynThreads, configured[2], st);
      return h4_launch<PAIR>(h4_synthesis_kernel<M, PAIR, H4Io::BF16>, p, kH4SynThreads, configured[3], st);
    } else {
      return -2;
    }
  }
  return h4_launch<PAIR>(h4_synthesis_kernel<M, PAIR, H4Io::F32>, p, kH4SynThreads, configured[0], st);
}

// ---------------------------------------------------------------------------------------------
// host: bank images, fp16 bits in UMMA K-major no-swizzle layout [chunk of 8 K][128 rows][8],
// rows = part * 64 + delta * M + (band | phase), part 0 = c1, part 1 = c2' = 2^11 (2^10 hk - c1)
// ---------------------------------------------------------------------------------------------
inline void hankel4_build_banks(const float* hk /*[M][L]*/, int M, int L, int jlo, int kt, uint16_t* img_analysis, uint16_t* img_synthesis) {
  auto bits = [](float v) {
    const __half h = __float2half_rn(v);
    uint16_t u;
    memcpy(&u, &h, 2);
    return u;
  };
  const int ks = (kt + 64 - M + 15) / 16, kp = 16 * ks;
  const int elo = jlo / M, ehi = (jlo + kt) / M - 1;
  const float sa = (float)(1 << kH16ScaleLog2), ss = (float)M * sa;
  for (int kc = 0; kc < kp / 8; ++kc)
    for (int row = 0; row < 128; ++row)
      for (int e8 = 0; e8 < 8; ++e8) {
        const int kap = 8 * kc + e8;
        const int part = row / 64, delta = (row % 64) / M, q = row % M;
        const size_t at = ((size_t)kc * 128 + row) * 8 + e8;
        {  // analysis: K index = tap offset within the (delta-shifted) window, q = band
          const int j = kap - M * delta;
          const float v = (j >= 0 && j < kt && jlo + j < L) ? sa * hk[(size_t)q * L + jlo + j] : 0.f;
          const float c1 = __half2float(__float2half_rn(v));
          img_analysis[at] = part == 0 ? bits(c1) : bits((v - c1) * kH4Res);
        }
        {  // synthesis: K index = (frame e, band kb) of the [frame][band] plane: lag = delta + ehi - e, tap M lag + q, q = output phase
          const int e = kap / M, kb = kap % M, lag = delta + ehi - e;
          const float v = (lag >= elo && lag <= ehi && M * lag + q < L) ? ss * hk[(size_t)kb * L + M * lag + q] : 0.f;
          const float c1 = __half2float(__float2half_rn(v));
          img_synthesis[at] = part == 0 ? bits(c1) : bits((v - c1) * kH4Res);
        }
      }
}

// per-rank images for the CTA-pair kernels: [rank][2 KS][96 rows][8]; rows 0-63 = rows 64 rank .. of the single-CTA image (rank 0:
// c1, rank 1: c2), rows 64-95 = c1 rows 32 rank .. 32 rank + 31 (this rank's half of the N = 64 operand)
inline void hankel4_pair_image(const uint16_t* single /*[2 KS][128][8]*/, int ks, uint16_t* pair /*[2][2 KS][96][8]*/) {
  const int chunks = 2 * ks;
  for (int r = 0; r < 2; ++r)
    for (int kc = 0; kc < chunks; ++kc)
      for (int row = 0; row < 96; ++row) {
        const int src = row < 64 ? 64 * r + row : 32 * r + (row - 64);
        memcpy(pair + (((size_t)r * chunks + kc) * 96 + row) * 8, single + ((size_t)kc * 128 + src) * 8, 16);
      }
}

// Largest number of edge K-steps (per side, <= max_trim) whose correction terms may be dropped: the dropped terms are bounded by
// 2 * 2^-11 * max|input| * (sum of the |bank| entries they multiply); returns the largest trim whose bound stays <= budget.
inline int hankel4_pick_trim(const float* hk /*[M][L]*/, int M, int L, int jlo, int kt, bool synthesis, double budget, int max_trim = 7) {
  const int ks = (kt + 64 - M + 15) / 16, fr = 64 / M, elo = jlo / M, ehi = (jlo + kt) / M - 1;
  int best = 0;
  for (int trim = 1; trim <= max_trim && ks - 2 * trim >= 1; ++trim) {
    double worst = 0.0;
    for (int delta = 0; delta < fr; ++delta)
      for (int q = 0; q < M; ++q) {  // q = band (analysis) or output phase (synthesis)
        double sum = 0.0;
        for (int side = 0; side < 2; ++side)
          for (int t = 0; t < trim; ++t) {
            const int s = side ? ks - 1 - t : t;
            for (int e16 = 0; e16 < 16; ++e16) {
              const int kap = 16 * s + e16;
              if (!synthesis) {
                const int j = kap - M * delta;
                if (j >= 0 && j < kt && jlo + j < L) sum += fabs((double)hk[(size_t)q * L + jlo + j]);
              } else {
                const int e = kap / M, kb = kap % M, lag = delta + ehi - e;
                if (lag >= elo && lag <= ehi && M * lag + q < L) sum += (double)M * fabs((double)hk[(size_t)kb * L + M * lag + q]);
              }
            }
          }
        worst = sum > worst ? sum : worst;
      }
    if (2.0 * worst / 2048.0 <= budget) best = trim;
    else break;
  }
  return best;
}

}  // namespace pqmf
