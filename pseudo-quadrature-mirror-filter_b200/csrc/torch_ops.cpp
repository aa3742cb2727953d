// torch custom ops `pqmf_b200::*` -- the glue between the Python mirror of the reference API
// (pqmf_b200/pqmf.py) and the C ABI (include/pqmf_b200.h).  Registered through the dispatcher
// with schemas so that torch.jit.script(...) of a module holding CachedPQMF works and a saved
// .ts loads wherever this library is loaded (the reference exports its wrappers that way:
// PQMFWrapper.py:102-108, PitchShifterPvoc/1-PitchShifterWrapper.py:337-343).
//
// There is deliberately NO CPU kernel: the ops are registered for the CUDA dispatch key only,
// so a CPU tensor raises "Could not run 'pqmf_b200::analysis' with arguments from the 'CPU'
// backend" instead of silently falling back.
#include <ATen/ATen.h>
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/csrc/autograd/custom_function.h>
#include <torch/library.h>

#include "../../include/pqmf_b200.h"

namespace {

void check_rc(int rc, const char* what) {
  TORCH_CHECK(rc == 0, what, " failed: ", pqmf_strerror(rc), " (code ", rc, ")");
}

void check_f32_cuda(const at::Tensor& t, const char* name) {
  TORCH_CHECK(t.is_cuda(), name, " must be a CUDA tensor (pqmf_b200 has no CPU fallback)");
  TORCH_CHECK(t.scalar_type() == at::kFloat, name, " must be float32, got ", t.scalar_type());
}

// element type of a signal / sub-band tensor of the offline ops: float32, or a half-precision type (the _x entry points of the C ABI)
int io_dtype(const at::Tensor& t, const char* name) {
  TORCH_CHECK(t.is_cuda(), name, " must be a CUDA tensor (pqmf_b200 has no CPU fallback)");
  switch (t.scalar_type()) {
    case at::kFloat: return PQMF_DTYPE_F32;
    case at::kHalf: return PQMF_DTYPE_F16;
    case at::kBFloat16: return PQMF_DTYPE_BF16;
    default: TORCH_CHECK(false, name, " must be float32, float16 or bfloat16, got ", t.scalar_type());
  }
  return -1;
}
// a half-precision call the library has no native kernel for (PQMF_ERR_UNSUPPORTED, nothing launched): the caller widens to fp32, runs
// the fp32 op and rounds the result -- bit-identical to the native path by construction
bool staged(int rc, int dtype) { return rc == PQMF_ERR_UNSUPPORTED && dtype != PQMF_DTYPE_F32; }

const float* tables_ptr(const at::Tensor& tables, const at::Tensor& like) {
  if (tables.numel() == 0) return nullptr;
  check_f32_cuda(tables, "tables");
  TORCH_CHECK(tables.is_contiguous() && tables.device() == like.device(), "tables must be contiguous and on the input's device");
  return tables.data_ptr<float>();
}

struct Bank {
  int64_t M, L;
  const float* ptr;
};

Bank bank_of(const at::Tensor& hk, const at::Tensor& like) {
  check_f32_cuda(hk, "hk");
  TORCH_CHECK(hk.dim() == 2 && hk.is_contiguous(), "hk must be a contiguous [n_band, L] tensor");
  TORCH_CHECK(hk.device() == like.device(), "hk and the input must be on the same device");
  return {hk.size(0), hk.size(1), hk.data_ptr<float>()};
}

// x [B, C, T] -> [B, C*M, n_frames]      (reference: C == 1; C > 1 is folded into the batch)
// float32 / float16 / bfloat16 in, the same type out
at::Tensor analysis(const at::Tensor& x, const at::Tensor& hk, const at::Tensor& tables, int64_t n_frames, int64_t flags) {
  const int dtype = io_dtype(x, "x");
  TORCH_CHECK(x.dim() == 3, "pqmf analysis expects [batch, channels, time], got ", x.dim(), " dims");
  const Bank bank = bank_of(hk, x);
  c10::cuda::CUDAGuard guard(x.device());
  const at::Tensor xc = x.contiguous();
  const int64_t B = xc.size(0) * xc.size(1), T = xc.size(2);
  TORCH_CHECK(n_frames >= 0 && B < (1LL << 31), "bad sizes");
  at::Tensor y = at::empty({xc.size(0), xc.size(1) * bank.M, n_frames}, xc.options());
  if (y.numel() == 0) return y;
  const int rc = pqmf_analysis_x(xc.data_ptr(), y.data_ptr(), bank.ptr, tables_ptr(tables, x), (int)B, (long)T, (long)n_frames, (int)bank.M,
                                 (int)bank.L, (unsigned)flags, dtype, (pqmf_stream_t)at::cuda::getCurrentCUDAStream().stream());
  if (staged(rc, dtype)) return analysis(xc.to(at::kFloat), hk, tables, n_frames, flags).to(x.scalar_type());
  check_rc(rc, "pqmf_analysis_x");
  return y;
}

// s [B, C*M, F] -> [B, C, M*F]
at::Tensor synthesis(const at::Tensor& s, const at::Tensor& hk, const at::Tensor& tables, int64_t delay_frames, int64_t flags) {
  const int dtype = io_dtype(s, "s");
  TORCH_CHECK(s.dim() == 3, "pqmf synthesis expects [batch, n_band, frames], got ", s.dim(), " dims");
  const Bank bank = bank_of(hk, s);
  TORCH_CHECK(s.size(1) % bank.M == 0, "sub-band tensor has ", s.size(1), " channels, expected a multiple of n_band=", bank.M);
  c10::cuda::CUDAGuard guard(s.device());
  const at::Tensor sc = s.contiguous();
  const int64_t C = sc.size(1) / bank.M, B = sc.size(0) * C, F = sc.size(2);
  TORCH_CHECK(B < (1LL << 31), "bad sizes");
  at::Tensor out = at::empty({sc.size(0), C, bank.M * F}, sc.options());
  if (out.numel() == 0) return out;
  const int rc = pqmf_synthesis_x(sc.data_ptr(), out.data_ptr(), bank.ptr, tables_ptr(tables, s), (int)B, (long)F, (int)bank.M, (int)bank.L,
                                  (int)delay_frames, (unsigned)flags, dtype, (pqmf_stream_t)at::cuda::getCurrentCUDAStream().stream());
  if (staged(rc, dtype)) return synthesis(sc.to(at::kFloat), hk, tables, delay_frames, flags).to(s.scalar_type());
  check_rc(rc, "pqmf_synthesis_x");
  return out;
}

// x [B, C, T] -> (out [B, C, M*n_frames], y [B, C*M, n_frames]): forward then inverse in one call (pqmf_roundtrip_f32)
std::tuple<at::Tensor, at::Tensor> roundtrip(const at::Tensor& x, const at::Tensor& hk, const at::Tensor& tables, int64_t n_frames,
                                             int64_t delay_frames, int64_t flags) {
  const int dtype = io_dtype(x, "x");
  TORCH_CHECK(x.dim() == 3, "pqmf roundtrip expects [batch, channels, time], got ", x.dim(), " dims");
  const Bank bank = bank_of(hk, x);
  c10::cuda::CUDAGuard guard(x.device());
  const at::Tensor xc = x.contiguous();
  const int64_t B = xc.size(0) * xc.size(1), T = xc.size(2);
  TORCH_CHECK(n_frames >= 0 && B < (1LL << 31), "bad sizes");
  at::Tensor y = at::empty({xc.size(0), xc.size(1) * bank.M, n_frames}, xc.options());
  at::Tensor out = at::empty({xc.size(0), xc.size(1), bank.M * n_frames}, xc.options());
  if (y.numel() == 0) return {out, y};
  const int rc = pqmf_roundtrip_x(xc.data_ptr(), y.data_ptr(), out.data_ptr(), bank.ptr, tables_ptr(tables, x), (int)B, (long)T, (long)n_frames,
                                  (int)bank.M, (int)bank.L, (int)delay_frames, (unsigned)flags, dtype,
                                  (pqmf_stream_t)at::cuda::getCurrentCUDAStream().stream());
  if (staged(rc, dtype)) {  // direction by direction (each native where it can be); the synthesis reads the rounded sub-bands
    at::Tensor ys = analysis(xc, hk, tables, n_frames, flags);
    return {synthesis(ys, hk, tables, delay_frames, flags), ys};
  }
  check_rc(rc, "pqmf_roundtrip_x");
  return {out, y};
}

// int16 PCM edge: pcm [B, T, C] interleaved WAV frames -> sub-bands [B, Cr * M, n_frames] (Cr = C, or 1 when down-mixing)
at::Tensor analysis_pcm16(const at::Tensor& pcm, const at::Tensor& hk, const at::Tensor& tables, int64_t n_frames, bool downmix, int64_t flags) {
  TORCH_CHECK(pcm.is_cuda(), "pcm must be a CUDA tensor (pqmf_b200 has no CPU fallback)");
  TORCH_CHECK(pcm.scalar_type() == at::kShort, "pcm must be int16, got ", pcm.scalar_type());
  TORCH_CHECK(pcm.dim() == 3, "pqmf analysis_pcm16 expects interleaved WAV frames [clips, time, channels], got ", pcm.dim(), " dims");
  const Bank bank = bank_of(hk, pcm);
  c10::cuda::CUDAGuard guard(pcm.device());
  const at::Tensor pc = pcm.contiguous();
  const int64_t B = pc.size(0), T = pc.size(1), C = pc.size(2), Cr = downmix ? 1 : C;
  TORCH_CHECK(n_frames >= 0 && B * C < (1LL << 31) && C >= 1 && C <= 64, "bad sizes");
  at::Tensor y = at::empty({B, Cr * bank.M, n_frames}, pc.options().dtype(at::kFloat));
  if (y.numel() == 0) return y;
  check_rc(pqmf_analysis_pcm16(pc.data_ptr<int16_t>(), y.data_ptr<float>(), bank.ptr, tables_ptr(tables, pcm), (int)B, (long)T, (int)C, downmix ? 1 : 0,
                               (long)n_frames, (int)bank.M, (int)bank.L, (unsigned)flags, (pqmf_stream_t)at::cuda::getCurrentCUDAStream().stream()),
           "pqmf_analysis_pcm16");
  return y;
}

// s [B, C * M, F] -> pcm [B, M * F, C] int16 (round to nearest even, saturating)
at::Tensor synthesis_pcm16(const at::Tensor& s, const at::Tensor& hk, const at::Tensor& tables, int64_t delay_frames, int64_t flags) {
  check_f32_cuda(s, "s");
  TORCH_CHECK(s.dim() == 3, "pqmf synthesis_pcm16 expects [batch, channels * n_band, frames], got ", s.dim(), " dims");
  const Bank bank = bank_of(hk, s);
  TORCH_CHECK(s.size(1) % bank.M == 0, "sub-band tensor has ", s.size(1), " channels, expected a multiple of n_band=", bank.M);
  c10::cuda::CUDAGuard guard(s.device());
  const at::Tensor sc = s.contiguous();
  const int64_t B = sc.size(0), C = sc.size(1) / bank.M, F = sc.size(2);
  TORCH_CHECK(B * C < (1LL << 31) && C >= 1 && C <= 64, "bad sizes");
  at::Tensor pcm = at::empty({B, bank.M * F, C}, sc.options().dtype(at::kShort));
  if (pcm.numel() == 0) return pcm;
  check_rc(pqmf_synthesis_pcm16(sc.data_ptr<float>(), pcm.data_ptr<int16_t>(), bank.ptr, tables_ptr(tables, s), (int)B, (int)C, (long)F, (int)bank.M,
                                (int)bank.L, (int)delay_frames, (unsigned)flags, (pqmf_stream_t)at::cuda::getCurrentCUDAStream().stream()),
           "pqmf_synthesis_pcm16");
  return pcm;
}

// x [B, C, T] -> out [B, C, M * n_frames] only (pqmf_reconstruct_f32): the sub-bands live in a scratch buffer of one row chunk
at::Tensor reconstruct(const at::Tensor& x, const at::Tensor& hk, const at::Tensor& tables, int64_t n_frames, int64_t delay_frames, int64_t flags) {
  const int dtype = io_dtype(x, "x");
  TORCH_CHECK(x.dim() == 3, "pqmf reconstruct expects [batch, channels, time], got ", x.dim(), " dims");
  const Bank bank = bank_of(hk, x);
  c10::cuda::CUDAGuard guard(x.device());
  const at::Tensor xc = x.contiguous();
  const int64_t B = xc.size(0) * xc.size(1), T = xc.size(2);
  TORCH_CHECK(n_frames >= 0 && B < (1LL << 31), "bad sizes");
  at::Tensor out = at::empty({xc.size(0), xc.size(1), bank.M * n_frames}, xc.options());
  if (out.numel() == 0) return out;
  const size_t bytes = pqmf_reconstruct_scratch_bytes((int)B, (long)T, (long)n_frames, (int)bank.M);
  at::Tensor scratch = at::empty({(int64_t)(bytes / sizeof(float))}, xc.options().dtype(at::kFloat));  // sized for fp32 sub-bands: holds either width
  const int rc = pqmf_reconstruct_x(xc.data_ptr(), out.data_ptr(), scratch.data_ptr(), bytes, bank.ptr, tables_ptr(tables, x), (int)B, (long)T,
                                    (long)n_frames, (int)bank.M, (int)bank.L, (int)delay_frames, (unsigned)flags, dtype,
                                    (pqmf_stream_t)at::cuda::getCurrentCUDAStream().stream());
  if (staged(rc, dtype)) {  // what process() computes: the synthesis of the rounded sub-bands
    scratch.reset();
    return synthesis(analysis(xc, hk, tables, n_frames, flags), hk, tables, delay_frames, flags);
  }
  check_rc(rc, "pqmf_reconstruct_x");
  return out;
}

// per-band hand-off (pqmf_synthesis_bands_f32): bands = n_band tensors [B, len_k]; returns (out [B, 1, M n_frames], new tail [M, Lx])
std::tuple<at::Tensor, at::Tensor> synthesis_bands(at::TensorList bands, const at::Tensor& hk, int64_t n_frames, int64_t delay_frames,
                                                   const at::Tensor& prev_tail, const at::Tensor& fade_out, const at::Tensor& fade_in, int64_t flags) {
  const Bank bank = bank_of(hk, hk);
  TORCH_CHECK((int64_t)bands.size() == bank.M, "expected ", bank.M, " band tensors, got ", bands.size());
  TORCH_CHECK(bank.M <= 64, "synthesis_bands supports n_band <= 64");
  c10::cuda::CUDAGuard guard(hk.device());
  std::vector<at::Tensor> keep;
  std::vector<const float*> ptrs;
  std::vector<long> lens;
  int64_t B = -1;
  for (const at::Tensor& b : bands) {
    check_f32_cuda(b, "band");
    TORCH_CHECK(b.dim() == 2 && b.device() == hk.device(), "every band must be a [batch, time] tensor on the bank's device");
    TORCH_CHECK(B < 0 || b.size(0) == B, "bands disagree on the batch size");
    B = b.size(0);
    keep.push_back(b.contiguous());
    ptrs.push_back(keep.back().data_ptr<float>());
    lens.push_back((long)b.size(1));
  }
  const int64_t Lx = prev_tail.numel() ? prev_tail.size(-1) : 0;
  const bool fade = Lx > 0;
  at::Tensor tail_out = at::empty_like(prev_tail);
  if (fade) {
    check_f32_cuda(prev_tail, "prev_tail");
    check_f32_cuda(fade_out, "fade_out");
    check_f32_cuda(fade_in, "fade_in");
    TORCH_CHECK(prev_tail.is_contiguous() && prev_tail.numel() == bank.M * Lx && fade_out.numel() == Lx && fade_in.numel() == Lx &&
                    fade_out.is_contiguous() && fade_in.is_contiguous(),
                "prev_tail must be [n_band, Lx] and fade_out / fade_in [Lx] (any leading singleton dims), contiguous");
  }
  at::Tensor out = at::empty({B, 1, bank.M * n_frames}, hk.options());
  check_rc(pqmf_synthesis_bands_f32(ptrs.data(), lens.data(), out.data_ptr<float>(), bank.ptr, (int)B, (long)n_frames, (int)bank.M, (int)bank.L,
                                    (int)delay_frames, fade ? prev_tail.data_ptr<float>() : nullptr, fade ? fade_out.data_ptr<float>() : nullptr,
                                    fade ? fade_in.data_ptr<float>() : nullptr, fade ? tail_out.data_ptr<float>() : nullptr, (int)Lx, (unsigned)flags,
                                    (pqmf_stream_t)at::cuda::getCurrentCUDAStream().stream()),
           "pqmf_synthesis_bands_f32");
  return {out, tail_out};
}

// streaming: state tensors are caller-owned ping-pong buffers; state_out is written in place.
at::Tensor analysis_stream(const at::Tensor& x, const at::Tensor& hk, const at::Tensor& tables, const at::Tensor& state_in,
                           at::Tensor state_out, int64_t frame_parity, int64_t flags) {
  check_f32_cuda(x, "x");
  check_f32_cuda(state_in, "state_in");
  check_f32_cuda(state_out, "state_out");
  TORCH_CHECK(x.dim() == 3, "pqmf streaming analysis expects [streams, channels, block], got ", x.dim(), " dims");
  const Bank bank = bank_of(hk, x);
  c10::cuda::CUDAGuard guard(x.device());
  const at::Tensor xc = x.contiguous();
  const int64_t B = xc.size(0) * xc.size(1), T = xc.size(2);
  TORCH_CHECK(T % bank.M == 0, "streaming block length ", T, " must be a multiple of n_band=", bank.M);
  TORCH_CHECK(state_in.is_contiguous() && state_out.is_contiguous() && state_in.numel() == B * bank.L &&
                  state_out.numel() == B * bank.L,
              "analysis state must be two contiguous [streams, L] buffers (L=", bank.L, ", streams=", B, ")");
  TORCH_CHECK(state_in.data_ptr() != state_out.data_ptr(), "state_in and state_out must not alias");
  at::Tensor y = at::empty({xc.size(0), xc.size(1) * bank.M, T / bank.M}, xc.options());
  if (B == 0) return y;
  check_rc(pqmf_analysis_stream_f32(xc.data_ptr<float>(), y.data_ptr<float>(), bank.ptr, tables_ptr(tables, x),
                                    state_in.data_ptr<float>(), state_out.data_ptr<float>(), (int)B, (long)T, (int)bank.M,
                                    (int)bank.L, (int)(frame_parity & 1), (unsigned)flags,
                                    (pqmf_stream_t)at::cuda::getCurrentCUDAStream().stream()),
           "pqmf_analysis_stream_f32");
  return y;
}

at::Tensor synthesis_stream(const at::Tensor& s, const at::Tensor& hk, const at::Tensor& tables, const at::Tensor& state_in,
                            at::Tensor state_out, int64_t frame_parity, int64_t flags) {
  check_f32_cuda(s, "s");
  check_f32_cuda(state_in, "state_in");
  check_f32_cuda(state_out, "state_out");
  TORCH_CHECK(s.dim() == 3, "pqmf streaming synthesis expects [streams, n_band, frames], got ", s.dim(), " dims");
  const Bank bank = bank_of(hk, s);
  TORCH_CHECK(s.size(1) % bank.M == 0, "sub-band tensor has ", s.size(1), " channels, expected a multiple of n_band=", bank.M);
  c10::cuda::CUDAGuard guard(s.device());
  const at::Tensor sc = s.contiguous();
  const int64_t C = sc.size(1) / bank.M, B = sc.size(0) * C, F = sc.size(2);
  TORCH_CHECK(state_in.is_contiguous() && state_out.is_contiguous() && state_in.numel() == B * bank.L &&
                  state_out.numel() == B * bank.L,
              "synthesis state must be two contiguous [streams, n_band, L/n_band] buffers");
  TORCH_CHECK(state_in.data_ptr() != state_out.data_ptr(), "state_in and state_out must not alias");
  TORCH_CHECK(F > 0, "empty block");
  at::Tensor out = at::empty({sc.size(0), C, bank.M * F}, sc.options());
  if (B == 0) return out;
  check_rc(pqmf_synthesis_stream_f32(sc.data_ptr<float>(), out.data_ptr<float>(), bank.ptr, tables_ptr(tables, s),
                                     state_in.data_ptr<float>(), state_out.data_ptr<float>(), (int)B, (long)F, (int)bank.M,
                                     (int)bank.L, (int)(frame_parity & 1), (unsigned)flags,
                                     (pqmf_stream_t)at::cuda::getCurrentCUDAStream().stream()),
           "pqmf_synthesis_stream_f32");
  return out;
}

// one streaming block step: (out, y) = (synthesis_stream(analysis_stream(x)), analysis_stream(x)), both states rolled
std::tuple<at::Tensor, at::Tensor> stream_step(const at::Tensor& x, const at::Tensor& hk, const at::Tensor& tables, const at::Tensor& xs_in,
                                               at::Tensor xs_out, const at::Tensor& ss_in, at::Tensor ss_out, int64_t parity_in, int64_t parity_out,
                                               int64_t flags) {
  check_f32_cuda(x, "x");
  const at::Tensor* states[4] = {&xs_in, &xs_out, &ss_in, &ss_out};
  for (const at::Tensor* t : states) check_f32_cuda(*t, "state");
  TORCH_CHECK(x.dim() == 3, "pqmf stream_step expects [streams, channels, block], got ", x.dim(), " dims");
  const Bank bank = bank_of(hk, x);
  c10::cuda::CUDAGuard guard(x.device());
  const at::Tensor xc = x.contiguous();
  const int64_t B = xc.size(0) * xc.size(1), T = xc.size(2);
  TORCH_CHECK(T > 0 && T % bank.M == 0, "streaming block length ", T, " must be a positive multiple of n_band=", bank.M);
  for (const at::Tensor* t : states)
    TORCH_CHECK(t->is_contiguous() && t->numel() == B * bank.L, "streaming state buffers must be contiguous with ", B * bank.L, " elements");
  TORCH_CHECK(xs_in.data_ptr() != xs_out.data_ptr() && ss_in.data_ptr() != ss_out.data_ptr(), "state_in and state_out must not alias");
  at::Tensor y = at::empty({xc.size(0), xc.size(1) * bank.M, T / bank.M}, xc.options());
  at::Tensor out = at::empty({xc.size(0), xc.size(1), T}, xc.options());
  if (B == 0) return {out, y};
  check_rc(pqmf_stream_step_f32(xc.data_ptr<float>(), y.data_ptr<float>(), out.data_ptr<float>(), bank.ptr, tables_ptr(tables, x), xs_in.data_ptr<float>(),
                                xs_out.data_ptr<float>(), ss_in.data_ptr<float>(), ss_out.data_ptr<float>(), (int)B, (long)T, (int)bank.M, (int)bank.L,
                                (int)(parity_in & 1), (int)(parity_out & 1), (unsigned)flags, (pqmf_stream_t)at::cuda::getCurrentCUDAStream().stream()),
           "pqmf_stream_step_f32");
  return {out, y};
}

// ---- stream pools (pqmf_stream_pool_*_f32): pool [2, P, ...] and phase [P] are mutated in place; ids is a CUDA int32 tensor of n
//      distinct stream numbers, trusted as it is (checking it would need a host synchronisation) ----
struct Pool {
  int64_t P;
  float* state;
  int* phase;
};
Pool pool_of(const at::Tensor& state, const at::Tensor& phase, const Bank& bank, const at::Tensor& like, const char* what) {
  check_f32_cuda(state, what);
  TORCH_CHECK(state.is_contiguous() && state.dim() >= 2 && state.size(0) == 2 && state.device() == like.device() &&
                  state.numel() == 2 * state.size(1) * bank.L,
              what, " must be a contiguous [2, P, ...] tensor of 2 * P * L float32 elements (L=", bank.L, ") on the input's device");
  TORCH_CHECK(phase.is_cuda() && phase.scalar_type() == at::kInt && phase.is_contiguous() && phase.dim() == 1 && phase.size(0) == state.size(1) &&
                  phase.device() == like.device(),
              "phase words must be a contiguous int32 [P] tensor on the input's device (P=", state.size(1), ")");
  TORCH_CHECK(state.size(1) >= 1 && state.size(1) < (1LL << 31), "bad pool size");
  return {state.size(1), state.data_ptr<float>(), phase.data_ptr<int>()};
}
const int* ids_of(const at::Tensor& ids, int64_t n, const at::Tensor& like) {
  TORCH_CHECK(ids.is_cuda() && ids.scalar_type() == at::kInt && ids.dim() == 1 && ids.is_contiguous() && ids.device() == like.device(),
              "ids must be a contiguous 1-D int32 CUDA tensor on the input's device");
  TORCH_CHECK(ids.size(0) == n, "ids has ", ids.size(0), " entries but the block has ", n, " rows");
  return ids.data_ptr<int>();
}

// x [n, 1, T] -> y [n, M, T / M]
at::Tensor stream_pool_analysis(const at::Tensor& x, const at::Tensor& hk, const at::Tensor& tables, at::Tensor xpool, at::Tensor xphase,
                                const at::Tensor& ids, int64_t flags) {
  check_f32_cuda(x, "x");
  TORCH_CHECK(x.dim() == 3 && x.size(1) == 1, "pqmf stream pool analysis expects [streams, 1, block], got ", x.sizes());
  const Bank bank = bank_of(hk, x);
  c10::cuda::CUDAGuard guard(x.device());
  const at::Tensor xc = x.contiguous();
  const int64_t n = xc.size(0), T = xc.size(2);
  TORCH_CHECK(T > 0 && T % bank.M == 0, "streaming block length ", T, " must be a positive multiple of n_band=", bank.M);
  const Pool pool = pool_of(xpool, xphase, bank, x, "xpool");
  const int* id = ids_of(ids, n, x);
  TORCH_CHECK(n <= pool.P, "more rows (", n, ") than streams in the pool (", pool.P, ")");
  at::Tensor y = at::empty({n, bank.M, T / bank.M}, xc.options());
  if (n == 0) return y;
  check_rc(pqmf_stream_pool_analysis_f32(xc.data_ptr<float>(), y.data_ptr<float>(), bank.ptr, tables_ptr(tables, x), pool.state, pool.phase, (int)pool.P,
                                         id, (int)n, (long)T, (int)bank.M, (int)bank.L, (unsigned)flags,
                                         (pqmf_stream_t)at::cuda::getCurrentCUDAStream().stream()),
           "pqmf_stream_pool_analysis_f32");
  return y;
}

// s [n, M, F] -> out [n, 1, M F]
at::Tensor stream_pool_synthesis(const at::Tensor& s, const at::Tensor& hk, const at::Tensor& tables, at::Tensor spool, at::Tensor sphase,
                                 const at::Tensor& ids, int64_t flags) {
  check_f32_cuda(s, "s");
  const Bank bank = bank_of(hk, s);
  TORCH_CHECK(s.dim() == 3 && s.size(1) == bank.M, "pqmf stream pool synthesis expects [streams, n_band, frames], got ", s.sizes());
  TORCH_CHECK(bank.L % bank.M == 0, "streaming synthesis needs L a multiple of n_band");
  c10::cuda::CUDAGuard guard(s.device());
  const at::Tensor sc = s.contiguous();
  const int64_t n = sc.size(0), F = sc.size(2);
  TORCH_CHECK(F > 0, "empty block");
  const Pool pool = pool_of(spool, sphase, bank, s, "spool");
  const int* id = ids_of(ids, n, s);
  TORCH_CHECK(n <= pool.P, "more rows (", n, ") than streams in the pool (", pool.P, ")");
  at::Tensor out = at::empty({n, 1, bank.M * F}, sc.options());
  if (n == 0) return out;
  check_rc(pqmf_stream_pool_synthesis_f32(sc.data_ptr<float>(), out.data_ptr<float>(), bank.ptr, tables_ptr(tables, s), pool.state, pool.phase,
                                          (int)pool.P, id, (int)n, (long)F, (int)bank.M, (int)bank.L, (unsigned)flags,
                                          (pqmf_stream_t)at::cuda::getCurrentCUDAStream().stream()),
           "pqmf_stream_pool_synthesis_f32");
  return out;
}

// one block step of the listed streams: (out [n, 1, T], y [n, M, T / M])
std::tuple<at::Tensor, at::Tensor> stream_pool_step(const at::Tensor& x, const at::Tensor& hk, const at::Tensor& tables, at::Tensor xpool,
                                                     at::Tensor xphase, at::Tensor spool, at::Tensor sphase, const at::Tensor& ids, int64_t flags) {
  check_f32_cuda(x, "x");
  TORCH_CHECK(x.dim() == 3 && x.size(1) == 1, "pqmf stream pool step expects [streams, 1, block], got ", x.sizes());
  const Bank bank = bank_of(hk, x);
  c10::cuda::CUDAGuard guard(x.device());
  const at::Tensor xc = x.contiguous();
  const int64_t n = xc.size(0), T = xc.size(2);
  TORCH_CHECK(T > 0 && T % bank.M == 0 && bank.L % bank.M == 0, "streaming block length ", T, " must be a positive multiple of n_band=", bank.M);
  const Pool xp = pool_of(xpool, xphase, bank, x, "xpool"), sp = pool_of(spool, sphase, bank, x, "spool");
  TORCH_CHECK(xp.P == sp.P, "the analysis and synthesis pools hold different numbers of streams");
  const int* id = ids_of(ids, n, x);
  TORCH_CHECK(n <= xp.P, "more rows (", n, ") than streams in the pool (", xp.P, ")");
  at::Tensor y = at::empty({n, bank.M, T / bank.M}, xc.options());
  at::Tensor out = at::empty({n, 1, T}, xc.options());
  if (n == 0) return {out, y};
  check_rc(pqmf_stream_pool_step_f32(xc.data_ptr<float>(), y.data_ptr<float>(), out.data_ptr<float>(), bank.ptr, tables_ptr(tables, x), xp.state, xp.phase,
                                     sp.state, sp.phase, (int)xp.P, id, (int)n, (long)T, (int)bank.M, (int)bank.L, (unsigned)flags,
                                     (pqmf_stream_t)at::cuda::getCurrentCUDAStream().stream()),
           "pqmf_stream_pool_step_f32");
  return {out, y};
}

// ---- int16 PCM blocks in the streaming ops (pqmf_*_stream_pcm16 / pqmf_stream_pool_*_pcm16): pcm [S, T, C] interleaved WAV frames, rows
//      S * C' (C' = 1 with downmix, else C; row s * C' + c = channel c of block s).  Where the library has no native kernel (PQMF_ERR_UNSUPPORTED,
//      nothing launched, no state touched) the op stages the call: widen, the fp32 op, quantise -- bit-identical to the native path by
//      construction ----
void check_pcm(const at::Tensor& pcm, const char* what) {
  TORCH_CHECK(pcm.is_cuda(), "pcm must be a CUDA tensor (pqmf_b200 has no CPU fallback)");
  TORCH_CHECK(pcm.scalar_type() == at::kShort, "pcm must be int16, got ", pcm.scalar_type());
  TORCH_CHECK(pcm.dim() == 3, "pqmf ", what, " expects interleaved int16 WAV frames [blocks, time, channels], got ", pcm.dim(), " dims");
  TORCH_CHECK(pcm.size(2) >= 1 && pcm.size(2) <= 64, "pqmf ", what, ": 1 to 64 channels, got ", pcm.size(2));
}
// [S, T, C] int16 -> [S, C', T] float32 with the kernels' arithmetic (pcm_sample): v / 32768, the down-mix summed in channel order, then / C
// (a tensor divisor: torch divides by a host scalar through its reciprocal, which is not the same rounding for C = 3, 5, ...)
at::Tensor pcm_widen(const at::Tensor& pcm, bool downmix) {
  const at::Tensor f = pcm.to(at::kFloat).mul_(1.0 / 32768.0);
  if (!downmix) return f.permute({0, 2, 1}).contiguous();
  at::Tensor acc = f.select(2, 0).clone();
  for (int64_t c = 1; c < f.size(2); ++c) acc.add_(f.select(2, c));
  return acc.div_(at::full({}, (double)f.size(2), acc.options())).unsqueeze(1);
}
// [S, C, T] float32 -> [S, T, C] int16: clamp(rint(v * 32768), -32768, 32767) (pcm_quantise)
at::Tensor pcm_quantise(const at::Tensor& v) {
  return at::clamp(at::round(v * 32768.0), -32768.0, 32767.0).to(at::kShort).permute({0, 2, 1}).contiguous();
}
pqmf_stream_t cur_stream() { return (pqmf_stream_t)at::cuda::getCurrentCUDAStream().stream(); }

// pcm [S, T, C] -> y [S, C' M, T / M]; state as analysis_stream (S C' streams)
at::Tensor analysis_stream_pcm16(const at::Tensor& pcm, const at::Tensor& hk, const at::Tensor& tables, const at::Tensor& state_in, at::Tensor state_out,
                                 int64_t frame_parity, bool downmix, int64_t flags) {
  check_pcm(pcm, "analysis_stream_pcm16");
  check_f32_cuda(state_in, "state_in");
  check_f32_cuda(state_out, "state_out");
  const Bank bank = bank_of(hk, pcm);
  c10::cuda::CUDAGuard guard(pcm.device());
  const at::Tensor pc = pcm.contiguous();
  const int64_t S = pc.size(0), T = pc.size(1), C = pc.size(2), Cr = downmix ? 1 : C, rows = S * Cr;
  TORCH_CHECK(rows < (1LL << 31), "bad sizes");
  TORCH_CHECK(T > 0 && T % bank.M == 0, "streaming block length ", T, " must be a positive multiple of n_band=", bank.M);
  TORCH_CHECK(state_in.is_contiguous() && state_out.is_contiguous() && state_in.numel() == rows * bank.L && state_out.numel() == rows * bank.L,
              "analysis state must be two contiguous [streams, L] buffers (L=", bank.L, ", streams=", rows, ")");
  TORCH_CHECK(state_in.data_ptr() != state_out.data_ptr(), "state_in and state_out must not alias");
  at::Tensor y = at::empty({S, Cr * bank.M, T / bank.M}, pc.options().dtype(at::kFloat));
  if (rows == 0) return y;
  const int rc = pqmf_analysis_stream_pcm16(pc.data_ptr<int16_t>(), y.data_ptr<float>(), bank.ptr, tables_ptr(tables, pcm), state_in.data_ptr<float>(),
                                            state_out.data_ptr<float>(), (int)S, (long)T, (int)C, downmix ? 1 : 0, (int)bank.M, (int)bank.L,
                                            (int)(frame_parity & 1), (unsigned)flags, cur_stream());
  if (rc == PQMF_ERR_UNSUPPORTED) return analysis_stream(pcm_widen(pc, downmix), hk, tables, state_in, state_out, frame_parity, flags);
  check_rc(rc, "pqmf_analysis_stream_pcm16");
  return y;
}

// s [S, C M, F] float32 -> pcm [S, M F, C] int16; state as synthesis_stream
at::Tensor synthesis_stream_pcm16(const at::Tensor& s, const at::Tensor& hk, const at::Tensor& tables, const at::Tensor& state_in, at::Tensor state_out,
                                  int64_t frame_parity, int64_t flags) {
  check_f32_cuda(s, "s");
  check_f32_cuda(state_in, "state_in");
  check_f32_cuda(state_out, "state_out");
  TORCH_CHECK(s.dim() == 3, "pqmf synthesis_stream_pcm16 expects [blocks, channels * n_band, frames], got ", s.dim(), " dims");
  const Bank bank = bank_of(hk, s);
  TORCH_CHECK(s.size(1) % bank.M == 0 && s.size(1) > 0, "sub-band tensor has ", s.size(1), " channels, expected a positive multiple of n_band=", bank.M);
  c10::cuda::CUDAGuard guard(s.device());
  const at::Tensor sc = s.contiguous();
  const int64_t S = sc.size(0), C = sc.size(1) / bank.M, F = sc.size(2), rows = S * C;
  TORCH_CHECK(C <= 64 && rows < (1LL << 31), "bad sizes");
  TORCH_CHECK(state_in.is_contiguous() && state_out.is_contiguous() && state_in.numel() == rows * bank.L && state_out.numel() == rows * bank.L,
              "synthesis state must be two contiguous [streams, n_band, L/n_band] buffers");
  TORCH_CHECK(state_in.data_ptr() != state_out.data_ptr(), "state_in and state_out must not alias");
  TORCH_CHECK(F > 0, "empty block");
  at::Tensor pcm = at::empty({S, bank.M * F, C}, sc.options().dtype(at::kShort));
  if (rows == 0) return pcm;
  const int rc = pqmf_synthesis_stream_pcm16(sc.data_ptr<float>(), pcm.data_ptr<int16_t>(), bank.ptr, tables_ptr(tables, s), state_in.data_ptr<float>(),
                                             state_out.data_ptr<float>(), (int)S, (int)C, (long)F, (int)bank.M, (int)bank.L, (int)(frame_parity & 1),
                                             (unsigned)flags, cur_stream());
  if (rc == PQMF_ERR_UNSUPPORTED) return pcm_quantise(synthesis_stream(sc, hk, tables, state_in, state_out, frame_parity, flags));
  check_rc(rc, "pqmf_synthesis_stream_pcm16");
  return pcm;
}

// one block step from PCM to PCM: (pcm_out [S, T, C'], y [S, C' M, T / M])
std::tuple<at::Tensor, at::Tensor> stream_step_pcm16(const at::Tensor& pcm, const at::Tensor& hk, const at::Tensor& tables, const at::Tensor& xs_in,
                                                     at::Tensor xs_out, const at::Tensor& ss_in, at::Tensor ss_out, int64_t parity_in, int64_t parity_out,
                                                     bool downmix, int64_t flags) {
  check_pcm(pcm, "stream_step_pcm16");
  const at::Tensor* states[4] = {&xs_in, &xs_out, &ss_in, &ss_out};
  for (const at::Tensor* t : states) check_f32_cuda(*t, "state");
  const Bank bank = bank_of(hk, pcm);
  c10::cuda::CUDAGuard guard(pcm.device());
  const at::Tensor pc = pcm.contiguous();
  const int64_t S = pc.size(0), T = pc.size(1), C = pc.size(2), Cr = downmix ? 1 : C, rows = S * Cr;
  TORCH_CHECK(rows < (1LL << 31), "bad sizes");
  TORCH_CHECK(T > 0 && T % bank.M == 0 && bank.L % bank.M == 0, "streaming block length ", T, " must be a positive multiple of n_band=", bank.M);
  for (const at::Tensor* t : states)
    TORCH_CHECK(t->is_contiguous() && t->numel() == rows * bank.L, "streaming state buffers must be contiguous with ", rows * bank.L, " elements");
  TORCH_CHECK(xs_in.data_ptr() != xs_out.data_ptr() && ss_in.data_ptr() != ss_out.data_ptr(), "state_in and state_out must not alias");
  at::Tensor y = at::empty({S, Cr * bank.M, T / bank.M}, pc.options().dtype(at::kFloat));
  at::Tensor out = at::empty({S, T, Cr}, pc.options());
  if (rows == 0) return {out, y};
  const int rc = pqmf_stream_step_pcm16(pc.data_ptr<int16_t>(), y.data_ptr<float>(), out.data_ptr<int16_t>(), bank.ptr, tables_ptr(tables, pcm),
                                        xs_in.data_ptr<float>(), xs_out.data_ptr<float>(), ss_in.data_ptr<float>(), ss_out.data_ptr<float>(), (int)S, (long)T,
                                        (int)C, downmix ? 1 : 0, (int)bank.M, (int)bank.L, (int)(parity_in & 1), (int)(parity_out & 1), (unsigned)flags,
                                        cur_stream());
  if (rc == PQMF_ERR_UNSUPPORTED) {  // direction by direction, each native where it can be
    at::Tensor ys = analysis_stream_pcm16(pc, hk, tables, xs_in, xs_out, parity_in, downmix, flags);
    return {synthesis_stream_pcm16(ys, hk, tables, ss_in, ss_out, parity_out, flags), ys};
  }
  check_rc(rc, "pqmf_stream_step_pcm16");
  return {out, y};
}

// pool: pcm [S, T, C] -> y [S, C' M, T / M]; ids [S C'] (row r is the next block of stream ids[r])
at::Tensor stream_pool_analysis_pcm16(const at::Tensor& pcm, const at::Tensor& hk, const at::Tensor& tables, at::Tensor xpool, at::Tensor xphase,
                                      const at::Tensor& ids, bool downmix, int64_t flags) {
  check_pcm(pcm, "stream pool analysis_pcm16");
  const Bank bank = bank_of(hk, pcm);
  c10::cuda::CUDAGuard guard(pcm.device());
  const at::Tensor pc = pcm.contiguous();
  const int64_t S = pc.size(0), T = pc.size(1), C = pc.size(2), Cr = downmix ? 1 : C, rows = S * Cr;
  TORCH_CHECK(T > 0 && T % bank.M == 0, "streaming block length ", T, " must be a positive multiple of n_band=", bank.M);
  const Pool pool = pool_of(xpool, xphase, bank, pcm, "xpool");
  const int* id = ids_of(ids, rows, pcm);
  TORCH_CHECK(rows <= pool.P, "more rows (", rows, ") than streams in the pool (", pool.P, ")");
  at::Tensor y = at::empty({S, Cr * bank.M, T / bank.M}, pc.options().dtype(at::kFloat));
  if (rows == 0) return y;
  const int rc = pqmf_stream_pool_analysis_pcm16(pc.data_ptr<int16_t>(), y.data_ptr<float>(), bank.ptr, tables_ptr(tables, pcm), pool.state, pool.phase,
                                                 (int)pool.P, id, (int)S, (long)T, (int)C, downmix ? 1 : 0, (int)bank.M, (int)bank.L, (unsigned)flags,
                                                 cur_stream());
  if (rc == PQMF_ERR_UNSUPPORTED)
    return stream_pool_analysis(pcm_widen(pc, downmix).view({rows, 1, T}), hk, tables, xpool, xphase, ids, flags).view({S, Cr * bank.M, T / bank.M});
  check_rc(rc, "pqmf_stream_pool_analysis_pcm16");
  return y;
}

// pool: s [S, C M, F] float32 -> pcm [S, M F, C] int16; ids [S C]
at::Tensor stream_pool_synthesis_pcm16(const at::Tensor& s, const at::Tensor& hk, const at::Tensor& tables, at::Tensor spool, at::Tensor sphase,
                                       const at::Tensor& ids, int64_t flags) {
  check_f32_cuda(s, "s");
  TORCH_CHECK(s.dim() == 3, "pqmf stream pool synthesis_pcm16 expects [blocks, channels * n_band, frames], got ", s.dim(), " dims");
  const Bank bank = bank_of(hk, s);
  TORCH_CHECK(s.size(1) % bank.M == 0 && s.size(1) > 0, "sub-band tensor has ", s.size(1), " channels, expected a positive multiple of n_band=", bank.M);
  TORCH_CHECK(bank.L % bank.M == 0, "streaming synthesis needs L a multiple of n_band");
  c10::cuda::CUDAGuard guard(s.device());
  const at::Tensor sc = s.contiguous();
  const int64_t S = sc.size(0), C = sc.size(1) / bank.M, F = sc.size(2), rows = S * C;
  TORCH_CHECK(C <= 64, "bad sizes");
  TORCH_CHECK(F > 0, "empty block");
  const Pool pool = pool_of(spool, sphase, bank, s, "spool");
  const int* id = ids_of(ids, rows, s);
  TORCH_CHECK(rows <= pool.P, "more rows (", rows, ") than streams in the pool (", pool.P, ")");
  at::Tensor pcm = at::empty({S, bank.M * F, C}, sc.options().dtype(at::kShort));
  if (rows == 0) return pcm;
  const int rc = pqmf_stream_pool_synthesis_pcm16(sc.data_ptr<float>(), pcm.data_ptr<int16_t>(), bank.ptr, tables_ptr(tables, s), pool.state, pool.phase,
                                                  (int)pool.P, id, (int)S, (int)C, (long)F, (int)bank.M, (int)bank.L, (unsigned)flags, cur_stream());
  if (rc == PQMF_ERR_UNSUPPORTED)
    return pcm_quantise(stream_pool_synthesis(sc.view({rows, bank.M, F}), hk, tables, spool, sphase, ids, flags).view({S, C, bank.M * F}));
  check_rc(rc, "pqmf_stream_pool_synthesis_pcm16");
  return pcm;
}

// pool: one block step from PCM to PCM of the listed streams: (pcm_out [S, T, C'], y [S, C' M, T / M])
std::tuple<at::Tensor, at::Tensor> stream_pool_step_pcm16(const at::Tensor& pcm, const at::Tensor& hk, const at::Tensor& tables, at::Tensor xpool,
                                                          at::Tensor xphase, at::Tensor spool, at::Tensor sphase, const at::Tensor& ids, bool downmix,
                                                          int64_t flags) {
  check_pcm(pcm, "stream pool step_pcm16");
  const Bank bank = bank_of(hk, pcm);
  c10::cuda::CUDAGuard guard(pcm.device());
  const at::Tensor pc = pcm.contiguous();
  const int64_t S = pc.size(0), T = pc.size(1), C = pc.size(2), Cr = downmix ? 1 : C, rows = S * Cr;
  TORCH_CHECK(T > 0 && T % bank.M == 0 && bank.L % bank.M == 0, "streaming block length ", T, " must be a positive multiple of n_band=", bank.M);
  const Pool xp = pool_of(xpool, xphase, bank, pcm, "xpool"), sp = pool_of(spool, sphase, bank, pcm, "spool");
  TORCH_CHECK(xp.P == sp.P, "the analysis and synthesis pools hold different numbers of streams");
  const int* id = ids_of(ids, rows, pcm);
  TORCH_CHECK(rows <= xp.P, "more rows (", rows, ") than streams in the pool (", xp.P, ")");
  at::Tensor y = at::empty({S, Cr * bank.M, T / bank.M}, pc.options().dtype(at::kFloat));
  at::Tensor out = at::empty({S, T, Cr}, pc.options());
  if (rows == 0) return {out, y};
  const int rc = pqmf_stream_pool_step_pcm16(pc.data_ptr<int16_t>(), y.data_ptr<float>(), out.data_ptr<int16_t>(), bank.ptr, tables_ptr(tables, pcm),
                                             xp.state, xp.phase, sp.state, sp.phase, (int)xp.P, id, (int)S, (long)T, (int)C, downmix ? 1 : 0, (int)bank.M,
                                             (int)bank.L, (unsigned)flags, cur_stream());
  if (rc == PQMF_ERR_UNSUPPORTED) {  // direction by direction, each native where it can be
    at::Tensor ys = stream_pool_analysis_pcm16(pc, hk, tables, xpool, xphase, ids, downmix, flags);
    return {stream_pool_synthesis_pcm16(ys, hk, tables, spool, sphase, ids, flags), ys};
  }
  check_rc(rc, "pqmf_stream_pool_step_pcm16");
  return {out, y};
}

int64_t launch_count() { return (int64_t)pqmf_launch_count(); }

// ---- autograd (SURVEY 8f-2: the reference path is differentiable, upstream users train through PQMF) --------------------
// Analysis and synthesis are each other's transposes up to the gain M and the frame delay, so both backward passes are the
// opposite-direction kernel with the same bank:
//   d/dx  analysis  : grad_x[t]   = sum_{k,n} sigma(k,n) gy[k,n] hk[k, t - nM + L/2]                 = synthesis(gy, delay 0)[t] / M
//   d/ds  synthesis : grad_s[k,n] = M sigma(k,n) sum_tau g[tau] hk[k, tau - (n + d) M + L/2] = M sigma(k,n) sigma(k,n+d) analysis(g)[k, n + d]
// (sigma(k,n) sigma(k,n+1) = (-1)^k; with PQMF_FLAG_NO_SIGN neither direction applies sigma and the factor is 1).
at::Tensor call_analysis(const at::Tensor& x, const at::Tensor& hk, const at::Tensor& tables, int64_t n_frames, int64_t flags) {
  static auto op = c10::Dispatcher::singleton().findSchemaOrThrow("pqmf_b200::analysis", "").typed<decltype(analysis)>();
  return op.call(x, hk, tables, n_frames, flags);
}
at::Tensor call_synthesis(const at::Tensor& s, const at::Tensor& hk, const at::Tensor& tables, int64_t delay_frames, int64_t flags) {
  static auto op = c10::Dispatcher::singleton().findSchemaOrThrow("pqmf_b200::synthesis", "").typed<decltype(synthesis)>();
  return op.call(s, hk, tables, delay_frames, flags);
}

// The tensor-core kernels carry every sample as two fp16 terms: full fp32-like accuracy for values of audio magnitude, but an
// ABSOLUTE error floor (~2^-36) below it and a range limit above (|v| < 65504).  Gradients have no natural scale (a mean-reduced
// loss gives 1e-7 .. 1e-9 per sample), so the backward passes normalise them by an exact power of two first: g' = g * 2^-e with
// e = floor(log2(max|g|)), computed on the device (no host sync), and fold 2^e into the constant the result is multiplied by anyway.
// With PQMF_FLAG_FP32 the kernels are plain fp32 and no scaling is needed.
struct GradScale {
  at::Tensor down, up;  // 0-dim fp32 tensors 2^-e, 2^e
};
// (the scale is computed in fp32 whatever g's type -- the clamp bounds do not exist in fp16 -- and multiplies g as a 0-dim tensor, so the
// scaled gradient keeps g's type)
GradScale grad_scale(const at::Tensor& g) {
  const at::Tensor amax = at::clamp(g.detach().abs().amax().to(at::kFloat), 1e-30, 1e30);
  const at::Tensor e = at::floor(at::log2(amax));
  return {at::exp2(-e), at::exp2(e)};
}

// The backward passes below normalise the gradient so that the kernels' outputs are near 1, and scale back afterwards.  In float32 and
// bfloat16 the scaling back is exact (fp32's exponent range); in float16 it can pass through the subnormal range, where a result already
// rounded at the kernel's output would lose bits.  So fp16 gradients are widened here and the fp32 result is rounded once at the end.
at::Tensor backward_in(const at::Tensor& g) { return g.scalar_type() == at::kHalf ? g.to(at::kFloat) : g; }

struct AnalysisFn : public torch::autograd::Function<AnalysisFn> {
  static at::Tensor forward(torch::autograd::AutogradContext* ctx, const at::Tensor& x, const at::Tensor& hk, const at::Tensor& tables,
                            int64_t n_frames, int64_t flags) {
    at::AutoDispatchBelowADInplaceOrView guard;
    ctx->save_for_backward({hk, tables});
    ctx->saved_data["T"] = x.size(-1);
    ctx->saved_data["flags"] = flags;
    return call_analysis(x, hk, tables, n_frames, flags);
  }
  static torch::autograd::variable_list backward(torch::autograd::AutogradContext* ctx, torch::autograd::variable_list grads) {
    const auto saved = ctx->get_saved_variables();
    const at::Tensor &hk = saved[0], &tables = saved[1];
    const int64_t T = ctx->saved_data["T"].toInt(), flags = ctx->saved_data["flags"].toInt(), M = hk.size(0);
    const auto dtype = grads[0].scalar_type();
    at::Tensor gy = backward_in(grads[0].contiguous());
    const int64_t F = gy.size(-1), need = (T + M - 1) / M;   // frames whose synthesis output covers [0, T)
    if (need > F) gy = at::constant_pad_nd(gy, {0, need - F});
    if (flags & PQMF_FLAG_FP32) {
      at::Tensor gx = call_synthesis(gy, hk, tables, 0, flags);
      return {(gx.slice(-1, 0, T) * (1.0 / (double)M)).to(dtype), at::Tensor(), at::Tensor(), at::Tensor(), at::Tensor()};
    }
    const GradScale sc = grad_scale(gy);
    at::Tensor gx = call_synthesis(gy * sc.down, hk, tables, 0, flags);
    gx = gx.slice(-1, 0, T) * (sc.up * (1.0 / (double)M));
    return {gx.to(dtype), at::Tensor(), at::Tensor(), at::Tensor(), at::Tensor()};
  }
};

struct SynthesisFn : public torch::autograd::Function<SynthesisFn> {
  static at::Tensor forward(torch::autograd::AutogradContext* ctx, const at::Tensor& s, const at::Tensor& hk, const at::Tensor& tables,
                            int64_t delay_frames, int64_t flags) {
    at::AutoDispatchBelowADInplaceOrView guard;
    ctx->save_for_backward({hk, tables});
    ctx->saved_data["delay"] = delay_frames;
    ctx->saved_data["flags"] = flags;
    return call_synthesis(s, hk, tables, delay_frames, flags);
  }
  static torch::autograd::variable_list backward(torch::autograd::AutogradContext* ctx, torch::autograd::variable_list grads) {
    const auto saved = ctx->get_saved_variables();
    const at::Tensor &hk = saved[0], &tables = saved[1];
    const int64_t d = ctx->saved_data["delay"].toInt(), flags = ctx->saved_data["flags"].toInt(), M = hk.size(0);
    const auto dtype = grads[0].scalar_type();
    const at::Tensor g = backward_in(grads[0].contiguous());          // [B, C, M F]
    const int64_t F = g.size(-1) / M;
    const bool plain = (flags & PQMF_FLAG_FP32) != 0;
    GradScale sc;
    if (!plain) sc = grad_scale(g);
    at::Tensor a = call_analysis(plain ? g : g * sc.down, hk, tables, F + d, flags);   // [B, C M, F + d]
    if (d > 0) {
      a = a.slice(-1, d, F + d);
      if (!(flags & PQMF_FLAG_NO_SIGN) && (d & 1)) {
        // counted in fp32 (bf16 cannot count past 256), applied in a's type
        const at::Tensor sign =
            (1.0 - 2.0 * at::arange(a.size(1), a.options().dtype(at::kFloat)).remainder((double)M).remainder(2.0)).to(a.scalar_type());
        a = a * sign.view({1, -1, 1});
      }
    }
    a = plain ? a * (double)M : a * (sc.up * (double)M);
    return {a.to(dtype), at::Tensor(), at::Tensor(), at::Tensor(), at::Tensor()};
  }
};

// the streaming ops mutate caller-owned state and have no backward: fail loudly instead of silently cutting the graph
at::Tensor analysis_stream_autograd(const at::Tensor& x, const at::Tensor& hk, const at::Tensor& tables, const at::Tensor& state_in,
                                    at::Tensor state_out, int64_t frame_parity, int64_t flags) {
  TORCH_CHECK(!(at::GradMode::is_enabled() && x.requires_grad()),
              "pqmf_b200::analysis_stream is not differentiable (streaming mode carries state across calls); use forward() for training "
              "or wrap the call in torch.no_grad()");
  at::AutoDispatchBelowADInplaceOrView guard;
  static auto op = c10::Dispatcher::singleton().findSchemaOrThrow("pqmf_b200::analysis_stream", "").typed<decltype(analysis_stream)>();
  return op.call(x, hk, tables, state_in, state_out, frame_parity, flags);
}
at::Tensor synthesis_stream_autograd(const at::Tensor& s, const at::Tensor& hk, const at::Tensor& tables, const at::Tensor& state_in,
                                     at::Tensor state_out, int64_t frame_parity, int64_t flags) {
  TORCH_CHECK(!(at::GradMode::is_enabled() && s.requires_grad()),
              "pqmf_b200::synthesis_stream is not differentiable (streaming mode carries state across calls); use inverse() for training "
              "or wrap the call in torch.no_grad()");
  at::AutoDispatchBelowADInplaceOrView guard;
  static auto op = c10::Dispatcher::singleton().findSchemaOrThrow("pqmf_b200::synthesis_stream", "").typed<decltype(synthesis_stream)>();
  return op.call(s, hk, tables, state_in, state_out, frame_parity, flags);
}

std::tuple<at::Tensor, at::Tensor> stream_step_autograd(const at::Tensor& x, const at::Tensor& hk, const at::Tensor& tables, const at::Tensor& xs_in,
                                                        at::Tensor xs_out, const at::Tensor& ss_in, at::Tensor ss_out, int64_t parity_in,
                                                        int64_t parity_out, int64_t flags) {
  TORCH_CHECK(!(at::GradMode::is_enabled() && x.requires_grad()),
              "pqmf_b200::stream_step is not differentiable (streaming mode carries state across calls); use forward() / inverse() for "
              "training or wrap the call in torch.no_grad()");
  at::AutoDispatchBelowADInplaceOrView guard;
  static auto op = c10::Dispatcher::singleton().findSchemaOrThrow("pqmf_b200::stream_step", "").typed<decltype(stream_step)>();
  return op.call(x, hk, tables, xs_in, xs_out, ss_in, ss_out, parity_in, parity_out, flags);
}

at::Tensor stream_pool_analysis_autograd(const at::Tensor& x, const at::Tensor& hk, const at::Tensor& tables, at::Tensor xpool, at::Tensor xphase,
                                         const at::Tensor& ids, int64_t flags) {
  TORCH_CHECK(!(at::GradMode::is_enabled() && x.requires_grad()),
              "pqmf_b200::stream_pool_analysis is not differentiable (a stream pool carries state across calls); use forward() for training "
              "or wrap the call in torch.no_grad()");
  at::AutoDispatchBelowADInplaceOrView guard;
  static auto op = c10::Dispatcher::singleton().findSchemaOrThrow("pqmf_b200::stream_pool_analysis", "").typed<decltype(stream_pool_analysis)>();
  return op.call(x, hk, tables, xpool, xphase, ids, flags);
}
at::Tensor stream_pool_synthesis_autograd(const at::Tensor& s, const at::Tensor& hk, const at::Tensor& tables, at::Tensor spool, at::Tensor sphase,
                                          const at::Tensor& ids, int64_t flags) {
  TORCH_CHECK(!(at::GradMode::is_enabled() && s.requires_grad()),
              "pqmf_b200::stream_pool_synthesis is not differentiable (a stream pool carries state across calls); use inverse() for training "
              "or wrap the call in torch.no_grad()");
  at::AutoDispatchBelowADInplaceOrView guard;
  static auto op = c10::Dispatcher::singleton().findSchemaOrThrow("pqmf_b200::stream_pool_synthesis", "").typed<decltype(stream_pool_synthesis)>();
  return op.call(s, hk, tables, spool, sphase, ids, flags);
}
std::tuple<at::Tensor, at::Tensor> stream_pool_step_autograd(const at::Tensor& x, const at::Tensor& hk, const at::Tensor& tables, at::Tensor xpool,
                                                             at::Tensor xphase, at::Tensor spool, at::Tensor sphase, const at::Tensor& ids,
                                                             int64_t flags) {
  TORCH_CHECK(!(at::GradMode::is_enabled() && x.requires_grad()),
              "pqmf_b200::stream_pool_step is not differentiable (a stream pool carries state across calls); use forward() / inverse() for "
              "training or wrap the call in torch.no_grad()");
  at::AutoDispatchBelowADInplaceOrView guard;
  static auto op = c10::Dispatcher::singleton().findSchemaOrThrow("pqmf_b200::stream_pool_step", "").typed<decltype(stream_pool_step)>();
  return op.call(x, hk, tables, xpool, xphase, spool, sphase, ids, flags);
}

at::Tensor synthesis_stream_pcm16_autograd(const at::Tensor& s, const at::Tensor& hk, const at::Tensor& tables, const at::Tensor& state_in,
                                           at::Tensor state_out, int64_t frame_parity, int64_t flags) {
  TORCH_CHECK(!(at::GradMode::is_enabled() && s.requires_grad()),
              "pqmf_b200::synthesis_stream_pcm16 is not differentiable (streaming mode carries state across calls, and int16 output has no "
              "gradient); use inverse() for training or wrap the call in torch.no_grad()");
  at::AutoDispatchBelowADInplaceOrView guard;
  static auto op = c10::Dispatcher::singleton().findSchemaOrThrow("pqmf_b200::synthesis_stream_pcm16", "").typed<decltype(synthesis_stream_pcm16)>();
  return op.call(s, hk, tables, state_in, state_out, frame_parity, flags);
}
at::Tensor stream_pool_synthesis_pcm16_autograd(const at::Tensor& s, const at::Tensor& hk, const at::Tensor& tables, at::Tensor spool, at::Tensor sphase,
                                                const at::Tensor& ids, int64_t flags) {
  TORCH_CHECK(!(at::GradMode::is_enabled() && s.requires_grad()),
              "pqmf_b200::stream_pool_synthesis_pcm16 is not differentiable (a stream pool carries state across calls, and int16 output has no "
              "gradient); use inverse() for training or wrap the call in torch.no_grad()");
  at::AutoDispatchBelowADInplaceOrView guard;
  static auto op =
      c10::Dispatcher::singleton().findSchemaOrThrow("pqmf_b200::stream_pool_synthesis_pcm16", "").typed<decltype(stream_pool_synthesis_pcm16)>();
  return op.call(s, hk, tables, spool, sphase, ids, flags);
}

at::Tensor analysis_autograd(const at::Tensor& x, const at::Tensor& hk, const at::Tensor& tables, int64_t n_frames, int64_t flags) {
  return AnalysisFn::apply(x, hk, tables, n_frames, flags);
}
at::Tensor synthesis_autograd(const at::Tensor& s, const at::Tensor& hk, const at::Tensor& tables, int64_t delay_frames, int64_t flags) {
  return SynthesisFn::apply(s, hk, tables, delay_frames, flags);
}

}  // namespace

TORCH_LIBRARY(pqmf_b200, m) {
  m.def("analysis(Tensor x, Tensor hk, Tensor tables, int n_frames, int flags) -> Tensor");
  m.def("synthesis(Tensor s, Tensor hk, Tensor tables, int delay_frames, int flags) -> Tensor");
  m.def(
      "analysis_stream(Tensor x, Tensor hk, Tensor tables, Tensor state_in, Tensor(a!) state_out, int frame_parity, int flags) "
      "-> Tensor");
  m.def(
      "synthesis_stream(Tensor s, Tensor hk, Tensor tables, Tensor state_in, Tensor(a!) state_out, int frame_parity, int flags) "
      "-> Tensor");
  m.def("roundtrip(Tensor x, Tensor hk, Tensor tables, int n_frames, int delay_frames, int flags) -> (Tensor, Tensor)");
  m.def(
      "stream_step(Tensor x, Tensor hk, Tensor tables, Tensor xs_in, Tensor(a!) xs_out, Tensor ss_in, Tensor(b!) ss_out, int parity_in, int parity_out, "
      "int flags) -> (Tensor, Tensor)");
  m.def("reconstruct(Tensor x, Tensor hk, Tensor tables, int n_frames, int delay_frames, int flags) -> Tensor");
  m.def("synthesis_bands(Tensor[] bands, Tensor hk, int n_frames, int delay_frames, Tensor prev_tail, Tensor fade_out, Tensor fade_in, int flags) -> (Tensor, Tensor)");
  m.def("analysis_pcm16(Tensor pcm, Tensor hk, Tensor tables, int n_frames, bool downmix, int flags) -> Tensor");
  m.def("synthesis_pcm16(Tensor s, Tensor hk, Tensor tables, int delay_frames, int flags) -> Tensor");
  m.def("stream_pool_analysis(Tensor x, Tensor hk, Tensor tables, Tensor(a!) xpool, Tensor(b!) xphase, Tensor ids, int flags) -> Tensor");
  m.def("stream_pool_synthesis(Tensor s, Tensor hk, Tensor tables, Tensor(a!) spool, Tensor(b!) sphase, Tensor ids, int flags) -> Tensor");
  m.def(
      "stream_pool_step(Tensor x, Tensor hk, Tensor tables, Tensor(a!) xpool, Tensor(b!) xphase, Tensor(c!) spool, Tensor(d!) sphase, Tensor ids, "
      "int flags) -> (Tensor, Tensor)");
  m.def(
      "analysis_stream_pcm16(Tensor pcm, Tensor hk, Tensor tables, Tensor state_in, Tensor(a!) state_out, int frame_parity, bool downmix, int flags) "
      "-> Tensor");
  m.def(
      "synthesis_stream_pcm16(Tensor s, Tensor hk, Tensor tables, Tensor state_in, Tensor(a!) state_out, int frame_parity, int flags) -> Tensor");
  m.def(
      "stream_step_pcm16(Tensor pcm, Tensor hk, Tensor tables, Tensor xs_in, Tensor(a!) xs_out, Tensor ss_in, Tensor(b!) ss_out, int parity_in, "
      "int parity_out, bool downmix, int flags) -> (Tensor, Tensor)");
  m.def(
      "stream_pool_analysis_pcm16(Tensor pcm, Tensor hk, Tensor tables, Tensor(a!) xpool, Tensor(b!) xphase, Tensor ids, bool downmix, int flags) "
      "-> Tensor");
  m.def("stream_pool_synthesis_pcm16(Tensor s, Tensor hk, Tensor tables, Tensor(a!) spool, Tensor(b!) sphase, Tensor ids, int flags) -> Tensor");
  m.def(
      "stream_pool_step_pcm16(Tensor pcm, Tensor hk, Tensor tables, Tensor(a!) xpool, Tensor(b!) xphase, Tensor(c!) spool, Tensor(d!) sphase, "
      "Tensor ids, bool downmix, int flags) -> (Tensor, Tensor)");
  m.def("launch_count() -> int", &launch_count);
}

TORCH_LIBRARY_IMPL(pqmf_b200, CUDA, m) {
  m.impl("analysis", &analysis);
  m.impl("synthesis", &synthesis);
  m.impl("analysis_stream", &analysis_stream);
  m.impl("synthesis_stream", &synthesis_stream);
  m.impl("roundtrip", &roundtrip);
  m.impl("stream_step", &stream_step);
  m.impl("reconstruct", &reconstruct);
  m.impl("synthesis_bands", &synthesis_bands);
  m.impl("analysis_pcm16", &analysis_pcm16);
  m.impl("synthesis_pcm16", &synthesis_pcm16);
  m.impl("stream_pool_analysis", &stream_pool_analysis);
  m.impl("stream_pool_synthesis", &stream_pool_synthesis);
  m.impl("stream_pool_step", &stream_pool_step);
  m.impl("analysis_stream_pcm16", &analysis_stream_pcm16);
  m.impl("synthesis_stream_pcm16", &synthesis_stream_pcm16);
  m.impl("stream_step_pcm16", &stream_step_pcm16);
  m.impl("stream_pool_analysis_pcm16", &stream_pool_analysis_pcm16);
  m.impl("stream_pool_synthesis_pcm16", &stream_pool_synthesis_pcm16);
  m.impl("stream_pool_step_pcm16", &stream_pool_step_pcm16);
}

// gradients w.r.t. the signal / the sub-bands only (the bank is a registered buffer in the reference, not a parameter)
TORCH_LIBRARY_IMPL(pqmf_b200, Autograd, m) {
  m.impl("analysis", &analysis_autograd);
  m.impl("synthesis", &synthesis_autograd);
  m.impl("analysis_stream", &analysis_stream_autograd);
  m.impl("synthesis_stream", &synthesis_stream_autograd);
  m.impl("stream_step", &stream_step_autograd);
  m.impl("stream_pool_analysis", &stream_pool_analysis_autograd);
  m.impl("stream_pool_synthesis", &stream_pool_synthesis_autograd);
  m.impl("stream_pool_step", &stream_pool_step_autograd);
  m.impl("synthesis_stream_pcm16", &synthesis_stream_pcm16_autograd);
  m.impl("stream_pool_synthesis_pcm16", &stream_pool_synthesis_pcm16_autograd);
}
