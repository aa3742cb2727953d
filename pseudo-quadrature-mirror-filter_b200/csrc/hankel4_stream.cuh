// Streaming (cached) blocks of n_band 8 / 16 / 32 on the Hankel-4 tensor-core kernels (hankel4.cuh).
//
// A streaming block is short (config 3: 2048 samples = 32 operand rows of 64 samples), so one 128-row MMA tile serves several
// streams.  Each stream gets its own REGION of plane rows: [history rows | block rows | padding to a multiple of 4 rows].  The
// causal window of block row i (analysis: samples 64 i - 448 .. 64 i - 64; synthesis: sub-band frames 4 i - 28 .. 4 i - 1)
// starts `hrows` rows before the row itself, i.e. at region row i -- so MMA row (region start + i) computes block row i with the
// UNCHANGED descriptors and bank images of the offline kernels, windows never leave their stream's region, and the MMA rows
// that fall on history / padding rows just compute values nobody stores (config 3: 3 streams per tile, 96 of 128 rows useful).
// The state is carried explicitly as in the fold kernels: the history rows are read from state_in, and the threads that load
// the tail of the block also write it to state_out (no separate roll).
//
// Stream pools (POOL instantiations, stream_pool.cuh): the state is a pool [2, P, ...] of P independent streams, and row r of the block
// is the next block of stream ids[r], whose phase word says which half holds its history and the parity of its next frame.  Each
// MMA row reads only its own stream's region, so which streams share a tile changes nothing: only the addresses of the history and
// of the roll, and the sign, come from ids and the phase word, loaded per tile one tile ahead with the block.  A row whose id is
// outside [0, P) is dead: zeros in, zeros out, no state touched.
#pragma once
#include <type_traits>

#include "hankel4.cuh"
#include "stream_pool.cuh"

namespace pqmf {

struct H4StreamGeom {
  int rows_b;  // block rows (64 samples / 4 frames each)
  int hrows;   // history rows in front of every block
  int pitch;   // region rows per stream: rows_b + hrows rounded up to a multiple of 4
  int spt;     // streams per tile = 128 / pitch
};
inline H4StreamGeom h4_stream_geom(long block_samples, int hist_samples) {
  H4StreamGeom s;
  s.rows_b = (int)(block_samples / 64);
  s.hrows = hist_samples / 64;
  s.pitch = (s.rows_b + s.hrows + 3) & ~3;
  s.spt = kH4Rows / s.pitch;
  return s;
}

struct H4AnalysisStreamParams {
  const float* x;         // [B, T]
  const float* hist_in;   // [B, L]: the L samples that preceded x
  float* hist_out;        // [B, L]: the last L samples of x (T >= L)
  float* y;               // [B, M, T / M]
  const uint16_t* bank;
  long T;
  int B, L;
  int parity, trim_lo, trim_hi;
  int pad_bytes;          // the region carries more history than the taps need (rounded up to whole rows): windows start this much later
  H4Shape g;
  H4StreamGeom s;
  long n_tiles;
};
// POOL: hist_in and hist_out are both the pool [2, P, L]
struct H4AnalysisStreamPoolParams : H4AnalysisStreamParams {
  StreamPoolIndex pool;
};

// streaming analysis: tiles blockIdx.x, + gridDim.x, ... of spt streams each
template <int M, bool POOL>
__global__ void __launch_bounds__(kH4Threads, 1)
    h4_analysis_stream_kernel(std::conditional_t<POOL, H4AnalysisStreamPoolParams, H4AnalysisStreamParams> p) {
  h4_kernel<true, kH4Workers>(p.g, p.bank, p.n_tiles, 1u, p.pad_bytes, p.trim_lo, p.trim_hi, [&](const H4Smem& sm, uint32_t tmem, uint32_t pfull_leader, unsigned n_iter) {
    constexpr int FR = 64 / M, HB = M / 2;  // frames per 64-sample row, bands per epilogue thread
    constexpr int NO = (kH4Rows * 8 + kH4Workers - 1) / kH4Workers;  // 4 x 8 samples per thread cover the 128 region rows of a tile
    const H4Shape& g = p.g;
    const H4StreamGeom& sg = p.s;
    const int tid = threadIdx.x;
    // rows past the last region are read by MMA rows whose results are never stored: make them finite once
    for (int u = sg.spt * sg.pitch * 32 + tid; u < g.rows * 32; u += kH4Workers)
#pragma unroll
      for (int pl = 0; pl < 4; ++pl) reinterpret_cast<float*>(sm.planes + pl * g.plane)[u] = 0.f;
    // tile-invariant plan of this thread's 8-sample groups, made once: the stream slot, RUNNING pointers to the group's source (history or
    // block) and -- for the groups that hold the tail of a block -- to its place in the next history, and what a tile step adds to them.
    // The loop below then only tests the slot against the live streams of the tile and bumps pointers (no per-tile index arithmetic).
    const int region_octs = sg.pitch * 8, n_octs = sg.spt * region_octs;
    const long F = p.T / M;
    const size_t step_x = (size_t)gridDim.x * sg.spt * p.T, step_h = (size_t)gridDim.x * sg.spt * p.L;
    constexpr int kDead = 1 << 20;  // slot of padding rows: never below the live-stream count
    int q_slot[NO];
    const float* src[NO];
    size_t src_step[NO];
    float* roll[NO];  // where the group goes in hist_out (nullptr: it is not part of the last L samples)
    int hofs[NO], rofs[NO];  // POOL: offset of a history group in its stream's pool row / of a roll group in the next history (-1: neither)
#pragma unroll
    for (int r = 0; r < NO; ++r) {
      const int u = tid + kH4Workers * r;
      q_slot[r] = kDead;
      src[r] = p.x;
      src_step[r] = 0;
      roll[r] = nullptr;
      hofs[r] = rofs[r] = -1;
      if (u < n_octs) {
        const int t = u / region_octs, w = u - t * region_octs, q = w >> 3, col = w & 7;
        const size_t stream0 = (size_t)blockIdx.x * sg.spt + t;  // the stream this group belongs to in this CTA's first tile
        if (q < sg.hrows) {
          q_slot[r] = t;
          if constexpr (POOL) {
            hofs[r] = (p.L - sg.hrows * 64) + q * 64 + 8 * col;
          } else {
            src[r] = p.hist_in + stream0 * p.L + ((p.L - sg.hrows * 64) + q * 64 + 8 * col);
            src_step[r] = step_h;
          }
        } else if (q - sg.hrows < sg.rows_b) {
          const long off = (q - sg.hrows) * 64 + 8 * col;
          q_slot[r] = t;
          src[r] = p.x + stream0 * p.T + off;
          src_step[r] = step_x;
          if (off >= p.T - p.L) {
            if constexpr (POOL) rofs[r] = (int)(off - (p.T - p.L));
            else roll[r] = p.hist_out + stream0 * p.L + (off - (p.T - p.L));
          }
        }
      }
    }
    float xr[NO][8];
    int nlive = 0;  // live streams of the tile held in xr
    int par_ld = 0, par_cur = 0, par_prev = 0;  // POOL: frame parity of this thread's drain row in the loaded / converted / drained tile
    auto load_tile = [&](long tile) {
      nlive = (int)min((long)sg.spt, (long)p.B - tile * sg.spt);
      if constexpr (POOL) {
        // the dependent index loads first (id, then its phase word); the data loads of history groups need both
        int id[NO], ph[NO];
#pragma unroll
        for (int r = 0; r < NO; ++r) {
          id[r] = q_slot[r] < nlive ? __ldg(p.pool.ids + tile * sg.spt + q_slot[r]) : -1;
          if ((unsigned)id[r] >= (unsigned)p.pool.P) id[r] = -1;  // dead row (or no stream): zeros, no roll
        }
        const int di = tid & 127, dt = di / sg.pitch;  // this thread's drain row (see drain below): region dt, block row di - dt pitch
        int did = dt < sg.spt && di - dt * sg.pitch < sg.rows_b && tile * sg.spt + dt < p.B ? __ldg(p.pool.ids + tile * sg.spt + dt) : -1;
        if ((unsigned)did >= (unsigned)p.pool.P) did = -1;
#pragma unroll
        for (int r = 0; r < NO; ++r) ph[r] = id[r] >= 0 ? __ldg(p.pool.phase + id[r]) : 0;
        par_ld = did >= 0 ? (__ldg(p.pool.phase + did) >> 1) & 1 : 0;
#pragma unroll
        for (int r = 0; r < NO; ++r) {
          const size_t row = (size_t)id[r];
          if (id[r] < 0) {
#pragma unroll
            for (int e = 0; e < 8; ++e) xr[r][e] = 0.f;
          } else if (hofs[r] >= 0) {
            ptx::ldg256_na(p.hist_in + ((size_t)(ph[r] & 1) * p.pool.P + row) * p.L + hofs[r], xr[r]);
          } else {
            ptx::ldg256_na(src[r], xr[r]);
          }
          src[r] += src_step[r];
          roll[r] = (rofs[r] >= 0 && id[r] >= 0) ? p.hist_out + ((size_t)(~ph[r] & 1) * p.pool.P + row) * p.L + rofs[r] : nullptr;
        }
      } else {
#pragma unroll
        for (int r = 0; r < NO; ++r) {
          if (q_slot[r] < nlive) {
            ptx::ldg256_na(src[r], xr[r]);
          } else {
#pragma unroll
            for (int e = 0; e < 8; ++e) xr[r][e] = 0.f;
          }
          src[r] += src_step[r];
        }
      }
    };
    // fp32 -> fp16 planes; the threads that hold the last L samples of a block also roll the history (here, where the data is
    // needed anyway: a store next to the load would make every prefetch wait for its own data)
    auto convert = [&](int pb) {
      unsigned char* p1 = sm.planes + (2 * pb) * g.plane;
      if constexpr (POOL) par_cur = par_ld;
#pragma unroll
      for (int r = 0; r < NO; ++r) {
        const int u = tid + kH4Workers * r;
        if (u < n_octs) {
          h4_split_store8(xr[r], p1, g.plane, sw128_offset((uint32_t)u * 16u));
          if (roll[r] != nullptr) {
            if (POOL || q_slot[r] < nlive) {  // POOL: load_tile set roll for live groups of this tile only
              *reinterpret_cast<float4*>(roll[r]) = make_float4(xr[r][0], xr[r][1], xr[r][2], xr[r][3]);
              *reinterpret_cast<float4*>(roll[r] + 4) = make_float4(xr[r][4], xr[r][5], xr[r][6], xr[r][7]);
            }
            if constexpr (!POOL) roll[r] += step_h;
          }
        }
      }
    };
    // D (TMEM) -> y: MMA row i = region t, row q: block row q (frames FR q .. FR q + FR - 1) of stream tile * spt + t when q < rows_b
    const int i = tid & 127, hb = tid >> 7;
    const int et = i / sg.pitch, eq = i - et * sg.pitch;
    const bool e_row = et < sg.spt && eq < sg.rows_b;
    float* yrun = p.y + (((size_t)blockIdx.x * sg.spt + et) * M + HB * hb) * F + FR * eq;  // this thread's rows of the CTA's first tile
    const size_t y_step = (size_t)gridDim.x * sg.spt * M * F;
    long tile = blockIdx.x, prev_tile = 0;
    auto drain = [&](int dbuf) {
      float v[FR][HB];
      h4_drain_analysis<M>(tmem, dbuf, tid, eq, POOL ? par_prev : p.parity, v);  // the first frame of block row eq is FR eq
      float* yp = yrun;
      yrun += y_step;
      if (!e_row || prev_tile * sg.spt + et >= p.B) return;
#pragma unroll
      for (int kk = 0; kk < HB; ++kk) {
        float w[FR];
#pragma unroll
        for (int dl = 0; dl < FR; ++dl) w[dl] = v[dl][kk];
        float* q = yp + (size_t)kk * F;
        if constexpr (FR >= 4) {
#pragma unroll
          for (int d4 = 0; d4 < FR; d4 += 4) __stcs(reinterpret_cast<float4*>(q + d4), make_float4(w[d4], w[d4 + 1], w[d4 + 2], w[d4 + 3]));
        } else if constexpr (FR == 2) {
          __stcs(reinterpret_cast<float2*>(q), make_float2(w[0], w[1]));
        } else {
          __stcs(q, w[0]);
        }
      }
    };

    load_tile(tile);
    h4_worker_loop<true>(sm, pfull_leader, n_iter, tid, convert, [&] { load_tile(tile + gridDim.x); }, drain, [&] {
      prev_tile = tile;
      tile += gridDim.x;
      if constexpr (POOL) par_prev = par_cur;
    } H4_TRACE(nullptr));
  } H4_TRACE(nullptr));
}

struct H4SynthesisStreamParams {
  const float* s;          // [B, M, F]
  const float* state_in;   // [B, M, K]: the K = L / M frames that preceded s
  float* state_out;        // [B, M, K]: the last K frames of s (F >= K)
  float* out;              // [B, M F]
  const uint16_t* bank;
  long F;
  int B, K;
  int parity, trim_lo, trim_hi;
  int pad_bytes;           // see H4AnalysisStreamParams
  H4Shape g;
  H4StreamGeom sg;
  long n_tiles;
};
// POOL: state_in and state_out are both the pool [2, P, M, K]
struct H4SynthesisStreamPoolParams : H4SynthesisStreamParams {
  StreamPoolIndex pool;
};

// streaming synthesis: tiles blockIdx.x, + gridDim.x, ... of spt streams each
template <int M, bool POOL>
__global__ void __launch_bounds__(kH4SynThreads, 1)
    h4_synthesis_stream_kernel(std::conditional_t<POOL, H4SynthesisStreamPoolParams, H4SynthesisStreamParams> p) {
  static_assert(M >= 8, "frame quads of 8-band groups (n_band 4 packs its chunks differently: offline kernels only)");
  h4_kernel<true, kH4SynWorkers>(p.g, p.bank, p.n_tiles, 1u, p.pad_bytes, p.trim_lo, p.trim_hi, [&](const H4Smem& sm, uint32_t tmem, uint32_t pfull_leader, unsigned n_iter) {
    constexpr int FR = 64 / M, NBG = M / 8;  // frames per 128-byte plane row, 8-band groups
    const H4Shape& g = p.g;
    const H4StreamGeom& sg = p.sg;
    const int tid = threadIdx.x, warp = tid >> 5;
    for (int u = sg.spt * sg.pitch * 32 + tid; u < g.rows * 32; u += kH4SynWorkers)
#pragma unroll
      for (int pl = 0; pl < 4; ++pl) reinterpret_cast<float*>(sm.planes + pl * g.plane)[u] = 0.f;
    // item (frame quad wq of the tile, band group bg): four frames x eight bands = four 16-byte chunks per plane.  A region holds
    // pitch * FR frames; its first hrows * FR frames are history (both multiples of 4: a quad never straddles the boundary)
    const int n_fq = sg.spt * sg.pitch * FR / 4;
    const int bg = tid / n_fq, wq = tid - bg * n_fq;
    const bool has_item = tid < NBG * n_fq;
    const int region_frames = sg.pitch * FR, hist_fr = sg.hrows * FR, block_fr = sg.rows_b * FR;
    const int lt = (4 * wq) / region_frames, lf = 4 * wq - lt * region_frames;  // region, first frame of the quad within the region
    const int fb = lf - hist_fr;  // first frame of this thread's quad within the block (negative: history)
    // tile-invariant plan, made once: RUNNING pointers to the quad's eight band rows (in the state for history frames, in s for block
    // frames), to its place in the next state when it is one of the block's last K frames, and what a tile step adds to them
    constexpr int kDead = 1 << 20;
    const size_t band0 = ((size_t)blockIdx.x * sg.spt + lt) * M + 8 * bg;  // first band row of the item in this CTA's first tile
    const size_t step_state = (size_t)gridDim.x * sg.spt * M * p.K;
    int slot = kDead;
    const float* src = p.s;
    size_t src_step = 0, src_pitch = 0;
    float* roll = nullptr;
    int hofs = -1, rofs = -1;  // POOL: offset of a history item in its stream's pool row [M, K] / of a roll item in the next history
    if (has_item) {
      if (fb < 0) {
        slot = lt;
        if constexpr (POOL) {
          hofs = 8 * bg * p.K + (p.K - hist_fr) + lf;
        } else {
          src = p.state_in + band0 * p.K + (p.K - hist_fr) + lf;
          src_step = step_state;
        }
        src_pitch = (size_t)p.K;
      } else if (fb < block_fr) {
        slot = lt;
        src = p.s + band0 * p.F + fb;
        src_step = (size_t)gridDim.x * sg.spt * M * p.F;
        src_pitch = (size_t)p.F;
        if (fb >= p.F - p.K) {  // the last K frames of the block become the next history
          if constexpr (POOL) rofs = 8 * bg * p.K + (fb - (p.F - p.K));
          else roll = p.state_out + band0 * p.K + (fb - (p.F - p.K));
        }
      }
    }
    float4 v[8];
    int nlive = 0;  // live streams of the tile held in v
    uint32_t flip_ld = 0;  // POOL: flip_even (below) of the stream of the loaded tile
    auto load_tile = [&](long tile) {
      nlive = (int)min((long)sg.spt, (long)p.B - tile * sg.spt);
      if constexpr (POOL) {
        int id = slot < nlive ? __ldg(p.pool.ids + tile * sg.spt + slot) : -1;
        if ((unsigned)id >= (unsigned)p.pool.P) id = -1;  // dead row (or no stream): zeros, no roll
        const int ph = id >= 0 ? __ldg(p.pool.phase + id) : 0;
        const size_t row = ((size_t)(ph & 1) * p.pool.P + (size_t)id) * M * p.K;  // the stream's current pool row; the next one is (ph & 1) ^ 1
        const float* from = hofs >= 0 ? p.state_in + row + hofs : src;
#pragma unroll
        for (int kk = 0; kk < 8; ++kk)
          v[kk] = id >= 0 ? ptx::ldg128_na(reinterpret_cast<const float4*>(from + (size_t)kk * src_pitch)) : make_float4(0.f, 0.f, 0.f, 0.f);
        src += src_step;
        roll = (rofs >= 0 && id >= 0) ? p.state_out + ((size_t)(~ph & 1) * p.pool.P + (size_t)id) * M * p.K + rofs : nullptr;
        flip_ld = (ph & 2) ? 0u : 0x80000000u;
      } else {
        const bool live = slot < nlive;
#pragma unroll
        for (int kk = 0; kk < 8; ++kk)
          v[kk] = live ? ptx::ldg128_na(reinterpret_cast<const float4*>(src + (size_t)kk * src_pitch)) : make_float4(0.f, 0.f, 0.f, 0.f);
        src += src_step;
      }
    };
    // sigma(k, n): odd bands flip on even global frames; regions and history lengths are multiples of 4 frames, so the parity is j's
    const uint32_t flip_even = (p.parity & 1) ? 0u : 0x80000000u, flip_odd = flip_even ^ 0x80000000u;
    auto convert = [&](int pb) {
      if (!has_item) return;
      unsigned char* p1 = sm.planes + (2 * pb) * g.plane;
      const uint32_t fe = POOL ? flip_ld : flip_even, fo = POOL ? flip_ld ^ 0x80000000u : flip_odd;
      if (roll != nullptr) {
        if (POOL || slot < nlive) {  // POOL: load_tile set roll for a live item of this tile only
#pragma unroll
          for (int kk = 0; kk < 8; ++kk) *reinterpret_cast<float4*>(roll + (size_t)kk * p.K) = v[kk];
        }
        if constexpr (!POOL) roll += step_state;
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float w[8];
        h4_synthesis_chunk8(v, j, (j & 1) ? fo : fe, w);
        h4_split_store8(w, p1, g.plane, sw128_offset((uint32_t)(4 * wq + j) * (2u * M) + 16u * bg));
      }
    };
    // D (TMEM) -> out (h4_drain_synthesis).  pitch and rows_b are multiples of 4, so the four rows of a lane quad belong to one region
    // and are valid or not together.
    const int i = tid & 127, hb = tid >> 7, lane = tid & 31;
    const int i0 = i & ~3, et = i0 / sg.pitch, eq0 = i0 - et * sg.pitch;
    const bool e_rows = et < sg.spt && eq0 < sg.rows_b;
    float* orun = p.out + ((size_t)blockIdx.x * sg.spt + et) * (size_t)(p.F * M) + 64 * eq0 + 32 * hb + 8 * (lane & 3);  // slot q: row eq0 + q of the block
    const size_t out_step = (size_t)gridDim.x * sg.spt * (size_t)(p.F * M);
    long tile = blockIdx.x, prev_tile = 0;
    auto drain = [&](int dbuf) {
      if (warp >= 8) return;  // every worker waited for the MMAs; the ninth warp has no TMEM rows to drain
      float val[4][8];
      h4_drain_synthesis(tmem, dbuf, tid, val);
      float* op = orun;
      orun += out_step;
      if (!e_rows || prev_tile * sg.spt + et >= p.B) return;
#pragma unroll
      for (int q = 0; q < 4; ++q) ptx::stg256_cs(op + (size_t)q * 64, val[q]);
    };

    load_tile(tile);
    h4_worker_loop<true>(sm, pfull_leader, n_iter, tid, convert, [&] { load_tile(tile + gridDim.x); }, drain, [&] {
      prev_tile = tile;
      tile += gridDim.x;
    } H4_TRACE(nullptr));
  } H4_TRACE(nullptr));
}

// launches (CTA pairs; on any error the caller runs other kernels: the fold kernels, or the direct form for pools)
// Params: H4AnalysisStreamParams, or H4AnalysisStreamPoolParams for the POOL instantiation
template <int M, typename Params>
inline int h4_launch_analysis_stream(Params p, cudaStream_t st) {
  constexpr bool POOL = std::is_same_v<Params, H4AnalysisStreamPoolParams>;
  static H4Configured configured;
  p.n_tiles = (p.B + p.s.spt - 1) / p.s.spt;
  return h4_launch<true>(h4_analysis_stream_kernel<M, POOL>, p, kH4Threads, configured, st);
}
// Params: H4SynthesisStreamParams, or H4SynthesisStreamPoolParams for the POOL instantiation
template <int M, typename Params>
inline int h4_launch_synthesis_stream(Params p, cudaStream_t st) {
  constexpr bool POOL = std::is_same_v<Params, H4SynthesisStreamPoolParams>;
  static H4Configured configured;
  p.n_tiles = (p.B + p.sg.spt - 1) / p.sg.spt;
  return h4_launch<true>(h4_synthesis_stream_kernel<M, POOL>, p, kH4SynThreads, configured, st);
}

}  // namespace pqmf
