/*
 * pqmf_b200 -- C ABI of the B200-native PQMF analysis / synthesis engine.
 *
 * This header is the drop-in boundary for the reference's hot path.  The reference
 * (oviniciuscesar/Pseudo-Quadrature-Mirror-Filter) has no FFI of its own: its boundary is
 * the Python module API of pqmf.py (class PQMF pqmf.py:202-288, class CachedPQMF
 * pqmf.py:306-354).  Each entry point below replaces the arithmetic behind one of those
 * methods; the Python mirror in pqmf_b200/pqmf.py (and the TORCH_LIBRARY ops in
 * csrc/torch_ops.cpp) call exactly these symbols and nothing else.  INTEGRATION.md shows
 * the binding a maintainer of the reference would add.
 *
 * Conventions
 *   - every data pointer is a DEVICE pointer to row-contiguous float32 unless the name ends
 *     in _host (host pointers) or _x (`void*` data of the element type `dtype`: float32, float16
 *     or bfloat16); the caller owns all buffers (including streaming state);
 *   - functions never allocate device memory, never synchronise, never throw: they enqueue
 *     on `stream` (a cudaStream_t passed as void*) and return 0 on success, a negative
 *     PQMF_ERR_* code for rejected arguments, or a positive cudaError_t value
 *     (pqmf_roundtrip_host_f32 is the exception: it owns a staging workspace and synchronises);
 *   - the tensor-core kernels represent every sample by two fp16 terms: |x|, |sub-band| < 65504;
 *   - M = n_band, L = hk.shape[1] (prototype length centre-padded to a power of two,
 *     pqmf.py:26-32), hk is the registered buffer `hk` [M, L] (pqmf.py:230);
 *   - sign mask sigma(k, n) = -1 iff band k is odd and GLOBAL frame index n is even
 *     (reverse_half, pqmf.py:13-22); `frame_parity` is (global index of the first frame) & 1.
 */
#ifndef PQMF_B200_H_
#define PQMF_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PQMF_B200_ABI_VERSION 2 /* 2: + pcm16, band table, reconstruct, multi-device host entry, PQMF_FLAG_FP32 */

#define PQMF_OK 0
#define PQMF_ERR_ARG (-1)         /* null pointer, non-positive size, misaligned buffer ...      */
#define PQMF_ERR_UNSUPPORTED (-2) /* combination the library has no kernel for                    */
#define PQMF_ERR_NO_DEVICE (-3)   /* no CUDA device / wrong architecture (needs sm_100)          */

/* flags (OR them; bits 8-23 are produced by pqmf_build_tables_f32 and belong to the tables they were returned with) */
#define PQMF_FLAG_EXACT 1u    /* every term of the registered hk: no fold factorisation, no trimmed correction steps.  Still the  *
                               * TENSOR-CORE kernels wherever they exist (Hankel kernels with trim 0 for large batches / many      *
                               * streams, Hankel-16 for small n_band 16 calls; the direct form elsewhere), i.e. samples are still  *
                               * carried as two fp16 terms (|x| < 65504).  PQMF_FLAG_FP32 is the plain-fp32 path.                  */
#define PQMF_FLAG_NO_SIGN 2u  /* skip sigma(k,n): the reference's free functions polyphase_forward / classic_* (pqmf.py:115-199) *
                               * leave reverse_half to the caller; offline only, runs the register-tiled direct form             */
#define PQMF_FLAG_FOLD 4u     /* n_band 16: force the fold + modulation kernels (measurement / debugging)                        */
#define PQMF_FLAG_FP32 16u    /* plain fp32 arithmetic on the CUDA cores (register-tiled direct form) for every shape: no fp16-pair   *
                               * representation of the samples, hence no range limit and fp32's relative accuracy at any signal     *
                               * level -- the arithmetic of the reference's conv1d, ~20x slower than the tensor-core kernels        */
#define PQMF_FLAG_NO_PAIR 8u  /* n_band 16: launch the Hankel kernels one CTA per SM instead of as CTA pairs (bit-identical)     */
#define PQMF_FLAG_NO_FOLD 32u /* n_band 16: never use the fold + modulation kernels (a bank that is not window x cosine: the     *
                               * Hankel kernels take hk as it is)                                                                */
#define PQMF_FLAG_TAPS(qlo, qn) (((unsigned)(qlo) << 8) | ((unsigned)(qn) << 12)) /* first kept tap / 32, kept taps / 32 */
/* edge K-steps (analysis, synthesis) of the Hankel kernels whose fp16 correction terms are provably below 6e-6 / 1.5e-5 of
 * max|input| for this bank and are skipped; 0 keeps every term */
#define PQMF_FLAG_H4_TRIM(ta, ts) ((((unsigned)(ta) & 7u) << 17) | ((((unsigned)(ta) >> 3) & 3u) << 24) | (((unsigned)(ts) & 7u) << 20))
#define PQMF_FLAG_H4_TRIM_A(flags) ((((flags) >> 17) & 7u) | ((((flags) >> 24) & 3u) << 3)) /* analysis: 0..31 (long banks: n_band 32 / 64) */
#define PQMF_FLAG_H4_TRIM_S(flags) (((flags) >> 20) & 7u)                                    /* synthesis: 0..7 */
/* the bank is too long for one SM's shared memory: the tables hold two tap ranges (TAPS describes one of them) that run as two
 * launches, the second accumulating into the output (n_band 64, long prototypes at n_band 32) */
#define PQMF_FLAG_H4_SPLIT (1u << 23)

typedef void* pqmf_stream_t; /* cudaStream_t */

int pqmf_abi_version(void);
const char* pqmf_strerror(int code);

/* Which kernel family a call with these parameters would use: 0 = register-tiled direct form (generic),
 * 1 = the tensor-core kernels: n_band 16 / L 512 (Hankel-4 offline, fold + modulation for streaming blocks and small
 * batches and few streams, Hankel-4 streaming for many streams) and n_band 4 / 8 / 32 / 64 (Hankel offline, large batches; n_band 8 / 32
 * also streaming with many streams).  PQMF_FLAG_FP32 and PQMF_FLAG_NO_SIGN always give 0.  `tables` may be NULL. */
int pqmf_path_for(int M, int L, const float* tables, unsigned flags);

/* ---- coefficient tables for the fast path (host side, one-off; replaces nothing in the reference:
 *      the reference re-derives its polyphase weights on every call, pqmf.py:128, :148-149) ----
 * Factorises hk[k, r + 2M q] ~= g[r + 2M q] * C[k, r] (SURVEY.md A.3) from the fp32 prototype h
 * (buffer `h`, pqmf.py:231) and returns the largest |hk - g (x) C| in *residual (may be NULL).
 * tables_host must hold pqmf_tables_numel(M, L) floats: [ g (L) | C_hi (M*2M) | C_lo (M*2M) ] followed by the fp16 images of
 * hk in the tensor cores' shared-memory operand layout (Hankel-16 and Hankel-4 kernels, analysis and synthesis).
 * *fast_flags (may be NULL) receives the PQMF_FLAG_TAPS(...) bits describing which taps are pure zero padding and the
 * PQMF_FLAG_H4_TRIM(...) bits; OR them into the `flags` of every compute call that is given these tables (the images are
 * built for exactly those taps: without the TAPS bits the offline Hankel kernels are not used).
 * Supported: n_band 16 / L 512 (all kernel families); n_band 4 / 8 / 16 / 32 / 64 with L = 16, 32 or 64 n_band (offline Hankel kernels).
 * Returns PQMF_ERR_UNSUPPORTED (and writes nothing) when (M, L) has no fast path or the bank does not fit one SM. */
long pqmf_tables_numel(int M, int L);
int pqmf_build_tables_f32(const float* hk_host, const float* h_host, int N, int M, int L, float* tables_host,
                          double* residual, unsigned* fast_flags);

/* ---- offline analysis: PQMF.forward (pqmf.py:247-259 -> polyphase_forward :115-130 /
 *      classic_forward :160-177, then reverse_half) and CachedPQMF.forward (:339-343) ----
 *   y[b,k,n] = sigma(k,n) * sum_j hk[k,j] * x[b, n*M + j - L/2],  x = 0 outside [0,T), 0 <= n < n_frames
 * x [B, T] -> y [B, M, n_frames].  n_frames = T/M (polyphase; requires T % M == 0 there),
 * floor(T/M) (classic) or ceil(T/M) (cached) -- the caller chooses. */
int pqmf_analysis_f32(const float* x, float* y, const float* hk, const float* tables, int B, long T, long n_frames, int M,
                      int L, unsigned flags, pqmf_stream_t stream);

/* ---- offline synthesis: PQMF.inverse (pqmf.py:272-288 -> reverse_half, polyphase_inverse :133-157 /
 *      classic_inverse :180-199) with delay_frames = 0, CachedPQMF.inverse (:345-354) with 1 ----
 *   out[b,tau] = M * sum_k sum_n sigma(k,n) s[b,k,n] * hk[k, tau - n*M + L/2 - delay_frames*M]
 * s [B, M, n_frames] -> out [B, M*n_frames]. */
int pqmf_synthesis_f32(const float* s, float* out, const float* hk, const float* tables, int B, long n_frames, int M, int L,
                       int delay_frames, unsigned flags, pqmf_stream_t stream);

/* ---- per-band hand-off of the pitch-shifter pipeline (SURVEY 8f-3; PitchShifterPvoc/1-PitchShifterWrapper.py:243-295: every
 *      sub-band goes through its own pitch shifter and comes back as a SEPARATE tensor of its own length; the reference then
 *      cross-fades each band's first Lx samples with the tail kept from the previous block (:259-276), centre-crops / zero-pads
 *      it to the analysis frame count (:279-289), concatenates the bands (:295) and calls CachedPQMF.inverse (:297)).
 * One synthesis call that reads the n_band tensors through a pointer table and applies cross-fade and crop / pad in its loads:
 *   bands   host array of M device pointers, band k = [B, lens[k]] row-contiguous;  lens  host array of M lengths
 *   s[b,k,f] = v_k[b, f + (lens[k] - n_frames) / 2]  (lens[k] > n_frames)   or   v_k[b, f - (n_frames - lens[k]) / 2], 0 outside
 *   v_k[b,u] = prev_tail[k,u] * fade_out[u] + band_k[b,u] * fade_in[u]  for u < Lx  (only when prev_tail != NULL, B == 1 and
 *              lens[k] >= Lx, as in the reference), band_k[b,u] otherwise
 *   out = pqmf_synthesis_f32(s, delay_frames);   tail_out[k,:] = v_k[0, lens[k]-Lx:]  (B == 1, lens[k] >= Lx), else prev_tail[k,:]
 * prev_tail / fade_out / fade_in / tail_out are device pointers ([M, Lx], [Lx], [Lx], [M, Lx]); tail_out must not alias
 * prev_tail.  M <= 64.  fp32 direct-form arithmetic (the hand-off is a real-time, batch-1 path). */
int pqmf_synthesis_bands_f32(const float* const* bands, const long* lens, float* out, const float* hk, int B, long n_frames, int M, int L,
                             int delay_frames, const float* prev_tail, const float* fade_out, const float* fade_in, float* tail_out, int Lx,
                             unsigned flags, pqmf_stream_t stream);

/* ---- int16 PCM edge (SURVEY 8f-4; the reference's inputs are the 16-bit WAVs under audio/, loaded by torchaudio.load as
 *      int16 / 32768 per channel: PQMFWrapper.py:113, 1-PitchShifterWrapper.py:348, PQMFPsWrapper.py:175; 2-TestBlocks.py:26-30
 *      down-mixes with mean(dim=0)).  The de-interleave and the int16 -> fp32 conversion happen inside the analysis loads, the
 *      fp32 -> int16 conversion and the interleave inside the synthesis stores: 2 B/sample/channel cross the API instead of 4. ----
 * pcm [B, T, C] interleaved WAV frames -> y [rows, M, n_frames], rows = B * C (row = clip * C + channel: torchaudio.load's [C, T]
 * per clip) or, with downmix != 0, rows = B and every row is the mean over the channels (fp32 sum in channel order, then / C).
 * Bit-identical to pqmf_analysis_f32 on the converted rows. */
int pqmf_analysis_pcm16(const int16_t* pcm, float* y, const float* hk, const float* tables, int B, long T, int C, int downmix,
                        long n_frames, int M, int L, unsigned flags, pqmf_stream_t stream);
/* s [B * C, M, n_frames] -> pcm [B, M * n_frames, C]: pqmf_synthesis_f32 followed by clamp(rint(v * 32768), -32768, 32767)
 * (round half to even, saturating), interleaved. */
int pqmf_synthesis_pcm16(const float* s, int16_t* pcm, const float* hk, const float* tables, int B, int C, long n_frames, int M, int L,
                         int delay_frames, unsigned flags, pqmf_stream_t stream);

/* ---- streaming (cached) mode: what cached_conv's cached padding does for the two layers
 *      CachedPQMF builds at pqmf.py:316-333 (SURVEY.md A.4), with explicit caller-owned state ----
 * analysis: frame n of the block sees samples [n*M - L, n*M) of (history ++ x):
 *   y[b,k,n] = sigma(k, n + frame_parity) * sum_j hk[k,j] * X[b, n*M + j - L]
 * state_in  [B, L]: the L samples that preceded x (zeros at stream start)
 * state_out [B, L]: the last L samples of (state_in ++ x); must not alias state_in.
 * T % M must be 0. */
int pqmf_analysis_stream_f32(const float* x, float* y, const float* hk, const float* tables, const float* state_in,
                             float* state_out, int B, long T, int M, int L, int frame_parity, unsigned flags,
                             pqmf_stream_t stream);

/* synthesis: output frame f of the block uses sub-band frames f-K .. f-1 of (history ++ s), K = L/M:
 *   out[b,tau] = M * sum_k sum_n sigma(k, n + frame_parity) S[b,k,n] * hk[k, tau - n*M - M]
 * state_in / state_out [B, M, K]: the K frames that preceded s / the last K frames of (state_in ++ s). */
int pqmf_synthesis_stream_f32(const float* s, float* out, const float* hk, const float* tables, const float* state_in,
                              float* state_out, int B, long n_frames, int M, int L, int frame_parity, unsigned flags,
                              pqmf_stream_t stream);

/* ---- one streaming block step: pqmf_analysis_stream_f32 followed by pqmf_synthesis_stream_f32 of the sub-bands it produced (what
 *      PQMFWrapper.process does per audio buffer in cached mode, PQMFWrapper.py:81-92), as ONE call (two launches on `stream`).
 *      x [B, T] -> y [B, M, T/M] and out [B, T]; xstate_* [B, L], sstate_* [B, M, L/M] as for the two entry points; parity_in /
 *      parity_out = global index & 1 of the first analysis frame / of the first sub-band frame fed to the synthesis. ---- */
int pqmf_stream_step_f32(const float* x, float* y, float* out, const float* hk, const float* tables, const float* xstate_in, float* xstate_out,
                         const float* sstate_in, float* sstate_out, int B, long T, int M, int L, int parity_in, int parity_out, unsigned flags,
                         pqmf_stream_t stream);

/* ---- stream pools: device-resident state of P independent streams, any n distinct of which are stepped by one call, in any order.
 *      Each stream has its own history, ping-pong half and frame parity, all on the device (caller-owned, fp32, zeros = P fresh streams):
 *        xpool [2, P, L]           analysis state;  spool [2, P, M, K], K = L / M   synthesis state
 *        xphase [P] / sphase [P]   one int32 word per stream and direction: bit 0 = the half that holds the stream's current history,
 *                                  bit 1 = the parity of the stream's next global frame index
 *      ids [n] (device int32, distinct, in [0, P)): row r of x [n, T] / y [n, M, T/M] / s / out [n, T] is the next block of stream ids[r].
 *      Per row the result is bit for bit that of pqmf_analysis_stream_f32 / pqmf_synthesis_stream_f32 with state_in = the stream's
 *      current half, state_out = its other half, frame_parity = its parity bit, run on the same kernel family: the streaming Hankel-4
 *      kernels exactly where a lockstep call with B = n runs them, the direct form everywhere else (also few-stream n_band 16, where a
 *      lockstep call runs the fold kernels).  After the compute launches, one more launch on `stream` flips the half bit of every listed
 *      stream and advances its parity by T / M (by n_frames for synthesis); streams not listed are untouched, state and phase word.
 *      A row whose id is outside [0, P) gives zeros and touches no state.  ids must be distinct; one pool is stepped from one stream at a
 *      time.  n == 0 returns 0.  The step runs both directions on the same ids (three launches). ---- */
int pqmf_stream_pool_analysis_f32(const float* x, float* y, const float* hk, const float* tables, float* xpool, int* xphase, int P,
                                  const int* ids, int n, long T, int M, int L, unsigned flags, pqmf_stream_t stream);
int pqmf_stream_pool_synthesis_f32(const float* s, float* out, const float* hk, const float* tables, float* spool, int* sphase, int P,
                                   const int* ids, int n, long n_frames, int M, int L, unsigned flags, pqmf_stream_t stream);
int pqmf_stream_pool_step_f32(const float* x, float* y, float* out, const float* hk, const float* tables, float* xpool, int* xphase,
                              float* spool, int* sphase, int P, const int* ids, int n, long T, int M, int L, unsigned flags,
                              pqmf_stream_t stream);

/* ---- grouped pool calls: sessions of different block lengths (a server whose clients choose their buffer sizes) stepped in one call.
 *      A group is n rows of one block length T (samples): ids [n] (device int32), x [n, T], y [n, M, T/M], out [n, T].  The analysis reads
 *      x and writes y, the synthesis reads y and writes out, the step does both; a pointer the direction does not use may be NULL.
 *      Up to 8 groups per call; ids distinct across ALL groups, at most P rows in total; n == 0 groups are allowed.  fp32 blocks here;
 *      int16 PCM and half-precision blocks in the _pcm16 and _x grouped entries below.
 *      Routing: the groups the streaming Hankel-4 kernels can plan (n_band 8 / 16 / 32, the block geometry, flags and alignment that a
 *      single-group call would need, whatever their own tile count) run together in ONE launch per direction followed by one phase-word
 *      launch, provided there are at least two of them and they make >= 96 tiles together (each direction, for a step).  Each of their rows
 *      is what the streaming Hankel-4 POOL kernels give for it: pqmf_stream_pool_*_f32 of that group whenever that call runs those kernels.
 *      Every other group runs through its pqmf_stream_pool_*_f32 entry with that entry's launches and bits.  G == 1 is that entry.  State
 *      halves and phase words are updated as by the single-group entries, each group's parity advanced by its own T / M; streams not
 *      listed are untouched.  All argument checks (PQMF_ERR_ARG) run on the host before anything is launched; G == 0 and all-empty
 *      calls return 0. ---- */
typedef struct pqmf_pool_group_f32 {
  const int* ids;
  int n;
  long T;
  const float* x;
  float* y;
  float* out;
} pqmf_pool_group_f32;
int pqmf_stream_pool_analysis_groups_f32(const pqmf_pool_group_f32* groups, int G, const float* hk, const float* tables, float* xpool, int* xphase,
                                         int P, int M, int L, unsigned flags, pqmf_stream_t stream);
int pqmf_stream_pool_synthesis_groups_f32(const pqmf_pool_group_f32* groups, int G, const float* hk, const float* tables, float* spool, int* sphase,
                                          int P, int M, int L, unsigned flags, pqmf_stream_t stream);
int pqmf_stream_pool_step_groups_f32(const pqmf_pool_group_f32* groups, int G, const float* hk, const float* tables, float* xpool, int* xphase,
                                     float* spool, int* sphase, int P, int M, int L, unsigned flags, pqmf_stream_t stream);

/* ---- int16 PCM blocks in the streaming calls (the PCM edge of pqmf_analysis_pcm16 / pqmf_synthesis_pcm16 on the streaming and pool entries
 *      above): what the reference's block driver streams (PitchShifterPvoc/2-TestBlocks.py:26-30) and what a server's sessions receive and
 *      return.  A PCM block is int16 interleaved WAV frames pcm [B, T, C]; widening is v / 32768 per channel, or with downmix != 0 the fp32
 *      sum over the channels in channel order, then / C; quantising is clamp(rint(v * 32768), -32768, 32767).  Rows are B * C (row
 *      b * C + c = channel c of clip b) or B with downmix.  Per row every entry is bit for bit its fp32 counterpart on the widened block,
 *      followed by quantising, with the same state and phase-word updates: PCM and fp32 blocks continue one stream.
 *        pqmf_analysis_stream_pcm16   pcm [B, T, C] -> y [rows, M, T/M]; state as pqmf_analysis_stream_f32 (rows streams)
 *        pqmf_synthesis_stream_pcm16  s [B * C, M, n_frames] -> pcm [B, M * n_frames, C]; state as pqmf_synthesis_stream_f32
 *        pqmf_stream_step_pcm16       pcm [B, T, C] -> y [rows, M, T/M] and pcm_out [B, T, C'] (C' = 1 with downmix, else C)
 *        pqmf_stream_pool_*_pcm16     the pool entries with PCM blocks: ids [rows] (row r is the next block of stream ids[r]), rows <= P
 *      Native kernels: the streaming Hankel-4 kernels (n_band 8 / 16 / 32), exactly where the fp32 call with the same rows, T, flags and
 *      pool-ness runs them and the PCM buffer is aligned for them (32 bytes in, 16 bytes out); PCM output natively for one channel per clip
 *      only.  Every other call (few streams, short or odd blocks, the fold / direct-form families, misaligned buffers, C' > 1 output)
 *      returns PQMF_ERR_UNSUPPORTED before anything is launched, with state and phase words untouched; the caller widens, calls the fp32
 *      entry and quantises (torch_ops.cpp does).  A step is native only when both directions are; a native step makes the launches of the
 *      fp32 step (two lockstep, three in a pool).  Argument errors are checked on the host first (PQMF_ERR_ARG; B == 0 returns 0). ---- */
int pqmf_analysis_stream_pcm16(const int16_t* pcm, float* y, const float* hk, const float* tables, const float* state_in, float* state_out, int B,
                               long T, int C, int downmix, int M, int L, int frame_parity, unsigned flags, pqmf_stream_t stream);
int pqmf_synthesis_stream_pcm16(const float* s, int16_t* pcm, const float* hk, const float* tables, const float* state_in, float* state_out, int B,
                                int C, long n_frames, int M, int L, int frame_parity, unsigned flags, pqmf_stream_t stream);
int pqmf_stream_step_pcm16(const int16_t* pcm, float* y, int16_t* pcm_out, const float* hk, const float* tables, const float* xstate_in,
                           float* xstate_out, const float* sstate_in, float* sstate_out, int B, long T, int C, int downmix, int M, int L, int parity_in,
                           int parity_out, unsigned flags, pqmf_stream_t stream);
int pqmf_stream_pool_analysis_pcm16(const int16_t* pcm, float* y, const float* hk, const float* tables, float* xpool, int* xphase, int P,
                                    const int* ids, int B, long T, int C, int downmix, int M, int L, unsigned flags, pqmf_stream_t stream);
int pqmf_stream_pool_synthesis_pcm16(const float* s, int16_t* pcm, const float* hk, const float* tables, float* spool, int* sphase, int P,
                                     const int* ids, int B, int C, long n_frames, int M, int L, unsigned flags, pqmf_stream_t stream);
int pqmf_stream_pool_step_pcm16(const int16_t* pcm, float* y, int16_t* pcm_out, const float* hk, const float* tables, float* xpool, int* xphase,
                                float* spool, int* sphase, int P, const int* ids, int B, long T, int C, int downmix, int M, int L, unsigned flags,
                                pqmf_stream_t stream);

/* ---- grouped pool calls with int16 PCM blocks: the grouped entries above (pqmf_stream_pool_*_groups_f32) with the PCM edge of the pool
 *      entries.  A group is n clips of C channels and T samples: ids [rows] (device int32; rows = n, or n * C without downmix; row s * C' + c
 *      is stream ids[s * C' + c]), pcm [n, T, C] interleaved WAV frames, y [n, C' M, T/M] and pcm_out [n, T, C'].  The analysis reads pcm and
 *      writes y, the synthesis reads y ([n, C M, T/M], rows n * C, no downmix) and writes pcm_out [n, T, C], the step does both; a pointer
 *      the direction does not use may be NULL.  downmix applies to the whole call; each group has its own T and C.  Per row the result is
 *      bit for bit pqmf_stream_pool_*_groups_f32 on the widened blocks followed by quantising, with the same pool and phase-word updates.
 *      Rule:
 *        1. All argument checks on the host first (PQMF_ERR_ARG): the single-group PCM pool entries' checks per group, 0 <= G <= 8, at most
 *           P rows in all, staged != NULL.  G == 0 and all-empty calls return 0.
 *        2. The joined groups are those the fp32 grouped call would join on freshly allocated widened blocks (the PCM buffers' alignment
 *           does not decide it).
 *        3. If a joined group cannot run natively (a PCM input not 32-byte aligned, C' > 1 output in a synthesis or step) or the first
 *           grouped launch does not start, the call returns PQMF_ERR_UNSUPPORTED with nothing launched: the caller widens every group,
 *           calls the fp32 grouped entry and quantises.  A step whose synthesis launch fails after its analysis ran returns
 *           cudaErrorLaunchFailure (a staged retry would step the analysis state twice).
 *        4. Otherwise one GROUPS PCM launch per direction and one phase-word launch for the joined groups, then every other group through
 *           its pqmf_stream_pool_*_pcm16 entry.  Where that entry refuses (PQMF_ERR_UNSUPPORTED, nothing launched), bit k of *staged is set
 *           and the call goes on; the caller then runs group k through the single-group pool calls on the widened block -- what the fp32
 *           grouped call does for a group it does not join.  *staged is 0 otherwise.  Returns 0.
 *      G == 1 is the group's pqmf_stream_pool_*_pcm16 entry (a refusal sets bit 0). ---- */
typedef struct pqmf_pool_group_pcm16 {
  const int* ids;
  int n;
  long T;
  int C;
  const int16_t* pcm;
  float* y;
  int16_t* pcm_out;
} pqmf_pool_group_pcm16;
int pqmf_stream_pool_analysis_groups_pcm16(const pqmf_pool_group_pcm16* groups, int G, int downmix, const float* hk, const float* tables,
                                           float* xpool, int* xphase, int P, int M, int L, unsigned flags, unsigned* staged, pqmf_stream_t stream);
int pqmf_stream_pool_synthesis_groups_pcm16(const pqmf_pool_group_pcm16* groups, int G, const float* hk, const float* tables, float* spool,
                                            int* sphase, int P, int M, int L, unsigned flags, unsigned* staged, pqmf_stream_t stream);
int pqmf_stream_pool_step_groups_pcm16(const pqmf_pool_group_pcm16* groups, int G, int downmix, const float* hk, const float* tables, float* xpool,
                                       int* xphase, float* spool, int* sphase, int P, int M, int L, unsigned flags, unsigned* staged,
                                       pqmf_stream_t stream);

/* ---- grouped pool calls with half-precision blocks: the grouped entries above (pqmf_stream_pool_*_groups_f32) with `void*` x, y and out
 *      whose element type is `dtype` (PQMF_DTYPE_*, see the half-precision pools below); the pool and phase words stay fp32 / int32.  With
 *      PQMF_DTYPE_F32 each one IS the _f32 grouped entry (and sets *staged = 0).  With PQMF_DTYPE_F16 / PQMF_DTYPE_BF16 per row the analysis
 *      is bit for bit pqmf_stream_pool_analysis_groups_f32 on the widened blocks followed by a round-to-nearest-even cast of y, the synthesis
 *      likewise on the widened sub-bands; pool halves and phase words are updated as by the fp32 call.  There is no grouped half step: a
 *      half step is the analysis followed by the synthesis of the ROUNDED sub-bands, and the two directions may join different groups.
 *      Rule, as for the PCM groups:
 *        1. All argument checks on the host first (PQMF_ERR_ARG): an unknown dtype, the single-group _x entries' checks per group,
 *           0 <= G <= 8, at most P rows in all, staged != NULL.  G == 0 and all-empty calls return 0.
 *        2. The joined groups are those the fp32 grouped call of the same direction would join on freshly allocated fp32 blocks and
 *           sub-bands (the half buffers' alignment does not decide it).
 *        3. If a joined group cannot run natively (a half x, y or out not 16-byte aligned) or the grouped launch does not start, the call
 *           returns PQMF_ERR_UNSUPPORTED with nothing launched: the caller widens every group, calls the fp32 grouped entry and rounds.
 *        4. Otherwise one GROUPS half launch and one phase-word launch for the joined groups, then every other group through its
 *           pqmf_stream_pool_*_x entry.  Where that entry refuses, bit k of *staged is set and the call goes on; the caller then runs group k
 *           through the single-group pool calls on the widened block.  *staged is 0 otherwise.  Returns 0.
 *      G == 1 is the group's pqmf_stream_pool_*_x entry (a refusal sets bit 0). ---- */
typedef struct pqmf_pool_group_x {
  const int* ids;
  int n;
  long T;
  const void* x;
  void* y;
  void* out;
} pqmf_pool_group_x;
int pqmf_stream_pool_analysis_groups_x(const pqmf_pool_group_x* groups, int G, const float* hk, const float* tables, float* xpool, int* xphase,
                                       int P, int M, int L, unsigned flags, int dtype, unsigned* staged, pqmf_stream_t stream);
int pqmf_stream_pool_synthesis_groups_x(const pqmf_pool_group_x* groups, int G, const float* hk, const float* tables, float* spool, int* sphase,
                                        int P, int M, int L, unsigned flags, int dtype, unsigned* staged, pqmf_stream_t stream);

/* ---- fused round trip on device buffers: PQMFWrapper.process (PQMFWrapper.py:81-92: forward, then inverse of the same
 *      sub-bands) and the Pvoc wrapper's forward (1-PitchShifterWrapper.py:303-316) ----
 * pqmf_analysis_f32 followed by pqmf_synthesis_f32 on the same stream, as one call; the synthesis kernels walk their tiles
 * last-to-first, so the most recently written part of y is still in L2 when it is read back.  x [B, T] -> y [B, M, n_frames]
 * (required: the sub-bands are an output of process()) and out [B, M * n_frames].  n_frames as for pqmf_analysis_f32. */
int pqmf_roundtrip_f32(const float* x, float* y, float* out, const float* hk, const float* tables, int B, long T, long n_frames,
                       int M, int L, int delay_frames, unsigned flags, pqmf_stream_t stream);

/* ---- reconstruction only: the forward of the Pvoc wrapper (1-PitchShifterWrapper.py:303-316: decompose, inverse, return the
 *      signal) never hands the sub-bands to anyone.  Here they are not an output either: they pass through `scratch`, row chunk
 *      by row chunk (<= 96 MB of sub-bands per chunk, >= 96 tiles when the batch allows), so that the synthesis launch of a chunk
 *      reads what the analysis launch just wrote from the 126 MB L2 and the next chunk overwrites the same lines before they are
 *      written back: less DRAM traffic than 16 B/sample and no [B, M, n_frames] allocation (4-13 % slower than pqmf_roundtrip_f32:
 *      the chunks cost launches).  Bit-identical to
 *      pqmf_roundtrip_f32's `out`.  scratch: device, >= pqmf_reconstruct_scratch_bytes(B, T, n_frames, M) bytes, caller-owned. */
size_t pqmf_reconstruct_scratch_bytes(int B, long T, long n_frames, int M);
int pqmf_reconstruct_f32(const float* x, float* out, float* scratch, size_t scratch_bytes, const float* hk, const float* tables, int B, long T,
                         long n_frames, int M, int L, int delay_frames, unsigned flags, pqmf_stream_t stream);

/* ---- half-precision signals and sub-bands (PyTorch's float16 / bfloat16 tensors) ----
 * pqmf_analysis_x, pqmf_synthesis_x, pqmf_roundtrip_x and pqmf_reconstruct_x are the _f32 entry points above with `void*` data
 * pointers whose element type is `dtype` (input and output alike).  With PQMF_DTYPE_F32 each one IS the _f32 entry.  With
 * PQMF_DTYPE_F16 / PQMF_DTYPE_BF16 the samples are widened to fp32 exactly in the kernels' loads, processed by the same kernels with
 * the same fp32 accumulation, and rounded to nearest even in the stores: bit-identical to the _f32 call on the widened input followed
 * by a round-to-nearest-even cast of its output, at half the bytes.  Native half-precision kernels exist for the offline Hankel-4
 * family only: a call runs natively where the _f32 call would run those kernels with an unsplit bank (no PQMF_FLAG_H4_SPLIT) as CTA
 * pairs, and its buffers are 16-byte aligned.  Every other call (small batches, ragged lengths, frame counts not a multiple of 4,
 * the fold / Hankel-16 / direct-form families, split banks, misaligned buffers) returns PQMF_ERR_UNSUPPORTED before anything is
 * launched; the caller then widens, calls the _f32 entry and rounds (torch_ops.cpp does).  pqmf_roundtrip_x and pqmf_reconstruct_x
 * run only when every launch they make is native.  pqmf_reconstruct_x's scratch is sized by pqmf_reconstruct_scratch_bytes. */
#define PQMF_DTYPE_F32 0
#define PQMF_DTYPE_F16 1
#define PQMF_DTYPE_BF16 2
int pqmf_analysis_x(const void* x, void* y, const float* hk, const float* tables, int B, long T, long n_frames, int M, int L, unsigned flags,
                    int dtype, pqmf_stream_t stream);
int pqmf_synthesis_x(const void* s, void* out, const float* hk, const float* tables, int B, long n_frames, int M, int L, int delay_frames,
                     unsigned flags, int dtype, pqmf_stream_t stream);
int pqmf_roundtrip_x(const void* x, void* y, void* out, const float* hk, const float* tables, int B, long T, long n_frames, int M, int L,
                     int delay_frames, unsigned flags, int dtype, pqmf_stream_t stream);
int pqmf_reconstruct_x(const void* x, void* out, void* scratch, size_t scratch_bytes, const float* hk, const float* tables, int B, long T,
                       long n_frames, int M, int L, int delay_frames, unsigned flags, int dtype, pqmf_stream_t stream);

/* ---- half-precision stream pools: pqmf_stream_pool_analysis_x / _synthesis_x / _step_x are the pool entries above
 *      (pqmf_stream_pool_*_f32) with `void*` blocks, sub-bands and outputs whose element type is `dtype`.  The pool (xpool, spool) and the
 *      phase words stay fp32 / int32 exactly as for the _f32 entries, so half, fp32 and PCM blocks continue one stream.  With
 *      PQMF_DTYPE_F32 each one IS the _f32 entry.  With PQMF_DTYPE_F16 / PQMF_DTYPE_BF16 per row the analysis is bit for bit the _f32
 *      analysis of the widened block followed by a round-to-nearest-even cast of y, the synthesis the _f32 synthesis of the widened
 *      sub-bands followed by the cast of out, and the step is the analysis followed by the synthesis of the ROUNDED y; pool halves and
 *      phase words are updated as by the _f32 entries.  Native kernels: the streaming Hankel-4 POOL kernels (n_band 8 / 16 / 32) with half
 *      loads and stores, exactly where the _f32 pool call with the same rows, T and flags runs them and the half buffers are 16-byte
 *      aligned.  Every other call (few streams, short or odd blocks, the direct form, split banks, misaligned buffers) returns
 *      PQMF_ERR_UNSUPPORTED before anything is launched, with pool and phase words untouched; the caller then widens, calls the _f32 entry
 *      and rounds, one direction at a time (torch_ops.cpp does).  The step is native only when both directions are (three launches, as the
 *      _f32 step).  Argument errors are checked on the host first (PQMF_ERR_ARG, also for an unknown dtype; n == 0 returns 0). ---- */
int pqmf_stream_pool_analysis_x(const void* x, void* y, const float* hk, const float* tables, float* xpool, int* xphase, int P, const int* ids,
                                int n, long T, int M, int L, unsigned flags, int dtype, pqmf_stream_t stream);
int pqmf_stream_pool_synthesis_x(const void* s, void* out, const float* hk, const float* tables, float* spool, int* sphase, int P, const int* ids,
                                 int n, long n_frames, int M, int L, unsigned flags, int dtype, pqmf_stream_t stream);
int pqmf_stream_pool_step_x(const void* x, void* y, void* out, const float* hk, const float* tables, float* xpool, int* xphase, float* spool,
                            int* sphase, int P, const int* ids, int n, long T, int M, int L, unsigned flags, int dtype, pqmf_stream_t stream);

/* ---- end-to-end host entry (what a non-torch host -- e.g. the Pure Data external that loads the
 *      reference's .ts, README.md:16 -- would call): host buffers in, host buffers out.
 * Pipelines H2D copy, analysis, synthesis and D2H copy over row chunks on internal streams and
 * synchronises before returning.  x_host [B, T] -> y_host [B, M, T/M] (may be NULL) and
 * out_host [B, T].  Pinned host buffers give full PCIe bandwidth; pageable ones work.
 * Tuning knobs (environment, read once per process): PQMF_HOST_CHUNK_MIB (row-chunk size in MiB of fp32 samples, default 8),
 * PQMF_HOST_SLOTS (chunks in flight, 2..8, default 4).  The per-device staging workspace (3 buffers per slot) is created on first use,
 * only grows, and is freed by pqmf_host_release(). */
int pqmf_roundtrip_host_f32(const float* x_host, float* y_host, float* out_host, const float* hk_host,
                            const float* tables_host, int B, long T, int M, int L, int delay_frames, unsigned flags,
                            int device);

/* The same with 16-bit PCM on both sides of the link (2 B/sample/channel each way instead of 4): pcm_host [B, T, C] interleaved WAV
 * frames -> y_host [B * C, M, T/M] (may be NULL) and out_host [B, T, C]; pqmf_analysis_pcm16 / pqmf_synthesis_pcm16 per chunk. */
int pqmf_roundtrip_host_pcm16(const int16_t* pcm_host, float* y_host, int16_t* out_host, const float* hk_host,
                              const float* tables_host, int B, long T, int C, int M, int L, int delay_frames, unsigned flags,
                              int device);

/* Multi-GPU host entry (SURVEY 8e: rows are independent, no collective): splits the B rows into n_devices contiguous shards (sizes
 * differing by at most one, in the order of `devices`) and runs pqmf_roundtrip_host_f32 for every shard concurrently, one host
 * thread and one staging workspace per device.  Returns the first non-zero status.  Calls for different devices never serialise
 * on each other (the workspace lock is per device). */
int pqmf_roundtrip_host_multi_f32(const float* x_host, float* y_host, float* out_host, const float* hk_host,
                                  const float* tables_host, int B, long T, int M, int L, int delay_frames, unsigned flags,
                                  const int* devices, int n_devices);
/* The row range [*start, *start + *count) of shard `shard` of `n_shards` (what pqmf_roundtrip_host_multi_f32 gives device number
 * `shard` of its list; host-only arithmetic, the same rule as the Python side's shard_rows). */
void pqmf_shard_rows(long n_rows, int n_shards, int shard, long* start, long* count);
/* The row-chunk schedule pqmf_roundtrip_host_f32 / _pcm16 use for B clips of C channels x T samples (host-only arithmetic): writes the
 * clips of the first max_chunks chunks to clips[] (may be NULL) and returns the number of chunks.  Every chunk holds whole clips, at
 * least the 96 tiles of 8192 samples the tensor-core kernels take (unless the whole call is smaller), at most one staging buffer. */
int pqmf_host_chunk_plan(int B, long T, int C, long* clips, int max_chunks);

/* Frees the per-device staging buffers / streams that the pqmf_roundtrip_host_* entry points keep between calls. */
void pqmf_host_release(void);

/* Number of kernels the library has launched in this process (bench.py reports it as gpu_launches). */
unsigned long long pqmf_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* PQMF_B200_H_ */
