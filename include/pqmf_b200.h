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
