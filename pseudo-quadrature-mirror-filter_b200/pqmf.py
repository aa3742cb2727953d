"""Drop-in mirror of the reference's ``pqmf.py`` module API, backed by the sm_100a kernels.

Same names, constructor arguments, buffers, attributes and error behaviour as the reference
(class PQMF pqmf.py:202-288, class CachedPQMF pqmf.py:306-354, free functions pqmf.py:13-199), so
``from pqmf import CachedPQMF`` / ``from PQMF.pqmf import CachedPQMF`` (see dropin/) keep working for
PQMFWrapper.py and both pitch-shifter wrappers.  What changes is where the arithmetic happens:
every ``forward`` / ``inverse`` is ONE fused kernel launch through ``torch.ops.pqmf_b200.*`` ->
C ABI (include/pqmf_b200.h) -> csrc/.  There is no CPU path: CPU tensors raise.

Differences that are deliberate (SURVEY.md A.6):
* 2-D inputs raise (the reference's 2-D branches are dead code: pqmf.py:248-249, :273-278);
* ``[B, C>1, T]`` is accepted and folded into the batch (the reference errors on it);
* both classes are TorchScript-scriptable (the reference's plain PQMF is not);
* ``CachedPQMF`` has an explicit streaming mode with caller-visible state instead of the hidden
  global switch of the third-party ``cached_conv`` package (``streaming=True`` / ``forward_stream``).

Precision: ``forward`` / ``inverse`` / ``process`` / ``reconstruct`` and the free functions accept float32, float16 and bfloat16
signals and sub-bands and return the input's dtype: ``forward(x_d)`` is bit-equal to ``forward(x_d.float()).to(d)`` (exact widening,
fp32 accumulation, round-to-nearest-even output; the large offline calls run on half-precision kernels, the rest widen, run the
fp32 kernels and round).  The input dtype and the module's dtype are independent: ``.half()`` / ``.to(torch.bfloat16)`` cast ``hk`` and
``h`` as the reference's module casts its buffers, and the arithmetic then uses that rounded bank, accumulated in fp32.  Other dtypes
(float64 included) raise.  The streaming, int16-PCM and per-band entry points take float32 sub-bands / signals only (the streaming calls
also take int16 PCM blocks: ``forward_stream_pcm16`` / ``inverse_stream_pcm16`` / ``process_stream_pcm16``).
"""
from __future__ import annotations

import math

from typing import List, Tuple

import torch
import torch.nn as nn

from . import _lib
from .design import center_pad_next_pow_2, get_prototype, get_qmf_bank, make_odd

_EMPTY = torch.zeros(0)
# fp32 buffers that are not numbers of the bank: module casts move them to the new device but never change their dtype (PQMF._apply)
_FP32_BUFFERS = ("_tables", "_x_state", "_s_state")

# largest |hk - g (x) C| accepted for the fold + modulation factorisation (SURVEY.md A.3: 1.7e-7 for the
# reference's own banks).  A bank that fails it (e.g. a hand-edited hk) silently uses the direct-form kernels.
_FOLD_RESIDUAL_LIMIT = 1e-6
assert _lib.PQMF_FLAG_FP32 == 16


def reverse_half(x: torch.Tensor) -> torch.Tensor:
    """Flip the sign of odd bands on even frames (reference pqmf.py:13-22).  Stand-alone helper only:
    inside the modules the mask is fused into the analysis store / synthesis load."""
    sign = torch.ones_like(x)
    sign[..., 1::2, ::2] = -1
    return x * sign


def _bank_2d(hk: torch.Tensor, rearrange_filter: bool, synthesis: bool) -> torch.Tensor:
    if rearrange_filter:
        return hk
    # caller passed the pre-arranged polyphase weights of the reference ("c (t m) -> c m t" for analysis,
    # flipped "c (t m) -> m c t" for synthesis, pqmf.py:128, :148-149); undo that to recover hk [M, L]
    if synthesis:
        m = hk.shape[1]
        return hk.permute(1, 2, 0).reshape(m, -1).flip(-1).contiguous()
    m = hk.shape[0]
    return hk.permute(0, 2, 1).reshape(m, -1).contiguous()


def polyphase_forward(x: torch.Tensor, hk: torch.Tensor, rearrange_filter: bool = True) -> torch.Tensor:
    """Analysis WITHOUT the sign mask (reference pqmf.py:115-130). x [B,1,T] -> [B,M,T/M]."""
    hk = _bank_2d(hk, rearrange_filter, False)
    if x.shape[-1] % hk.shape[0] != 0:
        raise RuntimeError(f"polyphase_forward: T={x.shape[-1]} is not a multiple of n_band={hk.shape[0]}")
    return torch.ops.pqmf_b200.analysis(x, hk.float(), _EMPTY, x.shape[-1] // hk.shape[0], _lib.PQMF_FLAG_NO_SIGN)


def classic_forward(x: torch.Tensor, hk: torch.Tensor) -> torch.Tensor:
    """Analysis WITHOUT the sign mask, any T (reference pqmf.py:160-177). x [B,1,T] -> [B,M,floor(T/M)]."""
    return torch.ops.pqmf_b200.analysis(x, hk.float(), _EMPTY, x.shape[-1] // hk.shape[0], _lib.PQMF_FLAG_NO_SIGN)


def polyphase_inverse(x: torch.Tensor, hk: torch.Tensor, rearrange_filter: bool = True) -> torch.Tensor:
    """Synthesis WITHOUT the sign mask (reference pqmf.py:133-157). x [B,M,F] -> [B,1,M*F]."""
    hk = _bank_2d(hk, rearrange_filter, True)
    return torch.ops.pqmf_b200.synthesis(x, hk.float(), _EMPTY, 0, _lib.PQMF_FLAG_NO_SIGN)


def classic_inverse(x: torch.Tensor, hk: torch.Tensor) -> torch.Tensor:
    """Synthesis WITHOUT the sign mask (reference pqmf.py:180-199; same function as polyphase_inverse)."""
    return torch.ops.pqmf_b200.synthesis(x, hk.float(), _EMPTY, 0, _lib.PQMF_FLAG_NO_SIGN)


def _refresh_after_load(module, _incompatible_keys):
    module.refresh_tables()


class PQMF(nn.Module):
    """Pseudo-QMF analysis / synthesis bank (reference pqmf.py:202-288).

    Parameters
    ----------
    attenuation : stop-band attenuation of the Kaiser prototype in dB (80 - 120)
    n_band      : number of sub-bands; must be a power of two when ``polyphase`` is True
    polyphase   : kept for API compatibility -- both settings run the same fused kernel and differ only in
                  the shape checks the reference applies (polyphase needs T % n_band == 0)
    n_channels  : stored, as in the reference; multichannel input is folded into the batch
    exact       : every term of the registered ``hk``: no fold factorisation and no trimmed correction steps.  Still the TENSOR-CORE
                  kernels wherever they exist (samples carried as two fp16 terms: |x| < 65504, absolute error floor ~1e-11)
    fp32        : plain fp32 arithmetic on the CUDA cores for every shape (the register-tiled direct form): the arithmetic of the
                  reference's ``conv1d`` -- no range limit, fp32's relative accuracy at any signal level, ~20x slower
    check_range : debug aid.  The tensor-core kernels assume audio-like magnitudes; with ``check_range=True`` every call first checks
                  max|x| (one host sync) and routes inputs beyond +-6e4 or entirely below 1e-6 to the fp32 kernels

    Signals and sub-bands may be float32, float16 or bfloat16; every output has its input's dtype (see the module docstring).
    """

    def __init__(self, attenuation, n_band, polyphase=True, n_channels=1, exact=False, fp32=False, check_range=False):
        super().__init__()
        proto = get_prototype(attenuation, n_band)
        if polyphase:
            power = math.log2(n_band)
            assert power == math.floor(power), "when using the polyphase algorithm, n_band must be a power of 2"
        h = torch.from_numpy(proto).float()
        hk = center_pad_next_pow_2(get_qmf_bank(h, n_band))
        self.register_buffer("hk", hk)
        self.register_buffer("h", h)
        self.register_buffer("_tables", torch.zeros(0), persistent=False)
        self.n_band: int = int(n_band)
        self.polyphase: bool = bool(polyphase)
        self.n_channels: int = int(n_channels)
        self._flags: int = (_lib.PQMF_FLAG_EXACT if exact else 0) | (_lib.PQMF_FLAG_FP32 if fp32 else 0)
        self.check_range: bool = bool(check_range)
        self.fold_residual: float = float("nan")
        self.refresh_tables()
        self.register_load_state_dict_post_hook(_refresh_after_load)

    def _apply(self, fn, recurse=True):
        """Module casts and moves.  ``hk`` and ``h`` follow a cast (``.half()``, ``.to(torch.bfloat16)``), as the reference's buffers
        do, and the tables are then re-derived from the bank as it now is.  The fp32 buffers that are not numbers of the bank follow
        the device only: ``_tables`` holds packed fp16 images, which a numeric cast would corrupt, and the streaming state stays fp32.
        A pure device move keeps the tables as they are (bit-equal, not rebuilt)."""
        hk_dtype = self.hk.dtype
        keep = {name: self._buffers[name] for name in _FP32_BUFFERS if self._buffers.get(name) is not None}
        super()._apply(fn, recurse)
        for name, buf in keep.items():
            moved = self._buffers[name]
            if moved is not None and moved.dtype != buf.dtype:
                self._buffers[name] = buf.to(moved.device)
        if self.hk.dtype != hk_dtype:
            self.refresh_tables()
        return self

    @torch.jit.unused
    def refresh_tables(self) -> None:
        """(Re)derive the fast-path coefficient tables from the current ``hk`` / ``h`` buffers (as fp32: the tables are always fp32)."""
        tables, residual, fast_flags = _lib.build_tables(self.hk, self.h)
        if tables.numel() and not (residual <= _FOLD_RESIDUAL_LIMIT):
            # bank is not window x cosine (e.g. a hand-edited hk was loaded): the fold + modulation kernels do not apply, the
            # Hankel kernels (which take hk as it is) still do
            fast_flags |= _lib.PQMF_FLAG_NO_FOLD
        self.fold_residual = residual
        self._flags = (self._flags & (_lib.PQMF_FLAG_EXACT | _lib.PQMF_FLAG_FP32)) | fast_flags
        self._tables = tables.to(self.hk.device)

    def _call_flags(self, x: torch.Tensor) -> int:
        """Flags for one call: with ``check_range`` inputs outside the comfortable range of the fp16-pair kernels go to fp32."""
        if self.check_range and x.numel() > 0:
            peak = float(x.detach().abs().amax().item())
            if not (1e-6 <= peak < 6.0e4):  # also catches inf / nan
                return self._flags | 16  # PQMF_FLAG_FP32 (a literal: TorchScript cannot close over module globals)
        return self._flags

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """x [B, 1, T] (or [B, C, T]) -> sub-bands [B, n_band, T / n_band] (or [B, C*n_band, ...])."""
        if x.dim() != 3:
            raise RuntimeError("PQMF.forward expects a 3-D tensor [batch, channels, time]; add the missing axes "
                               "(the reference's 2-D branch is dead code)")
        if self.n_band == 1:
            return x
        t = x.shape[-1]
        if self.polyphase and t % self.n_band != 0:
            raise RuntimeError("polyphase PQMF needs the number of samples to be a multiple of n_band")
        return torch.ops.pqmf_b200.analysis(x, self.hk.float(), self._tables, t // self.n_band, self._call_flags(x))

    @torch.jit.export
    def inverse(self, x: torch.Tensor) -> torch.Tensor:
        """sub-bands [B, n_band, F] -> signal [B, 1, n_band * F]."""
        if x.dim() != 3:
            raise RuntimeError("PQMF.inverse expects a 3-D tensor [batch, n_band, frames]")
        if self.n_band == 1:
            return x
        return torch.ops.pqmf_b200.synthesis(x, self.hk.float(), self._tables, 0, self._call_flags(x))

    @torch.jit.export
    def reconstruct(self, x: torch.Tensor) -> torch.Tensor:
        """``inverse(forward(x))`` when nobody needs the sub-bands -- the ``forward`` of the reference's Pvoc wrapper
        (``1-PitchShifterWrapper.py:303-316``).  The sub-bands go through an L2-sized scratch buffer chunk by chunk instead of a
        ``[B, n_band, T / n_band]`` tensor: no sub-band allocation and less DRAM traffic than ``process`` (a few per cent slower: the
        row chunks cost launches); the same bits."""
        if x.dim() != 3:
            raise RuntimeError("reconstruct expects a 3-D tensor [batch, channels, time]")
        if self.n_band == 1:
            return x
        if torch.is_grad_enabled() and x.requires_grad:
            return self.inverse(self.forward(x))
        return torch.ops.pqmf_b200.reconstruct(x, self.hk.float(), self._tables, self._n_frames_of(x.shape[-1]), self._inverse_delay(), self._flags)

    def _n_frames_of(self, t: int) -> int:
        if self.polyphase and t % self.n_band != 0:
            raise RuntimeError("polyphase PQMF needs the number of samples to be a multiple of n_band")
        return t // self.n_band

    @torch.jit.export
    def forward_pcm16(self, pcm: torch.Tensor, downmix: bool = False) -> torch.Tensor:
        """Analysis straight from 16-bit PCM (SURVEY 8f-4): ``pcm`` int16 ``[clips, time, channels]`` (interleaved WAV frames) ->
        sub-bands ``[clips, channels * n_band, time / n_band]``, bit-identical to ``forward(pcm.transpose(1, 2) / 32768)`` -- what
        ``torchaudio.load`` + ``forward`` give in the reference's scripts -- with the de-interleave and the conversion fused into the
        kernel's loads.  ``downmix=True``: one row per clip, the mean over the channels (``2-TestBlocks.py:26-30``)."""
        if pcm.dim() != 3:
            raise RuntimeError("forward_pcm16 expects int16 WAV frames [clips, time, channels]")
        t = pcm.shape[1]
        if self.polyphase and t % self.n_band != 0:
            raise RuntimeError("polyphase PQMF needs the number of samples to be a multiple of n_band")
        return torch.ops.pqmf_b200.analysis_pcm16(pcm, self.hk.float(), self._tables, t // self.n_band, downmix, self._flags)

    @torch.jit.export
    def inverse_pcm16(self, x: torch.Tensor) -> torch.Tensor:
        """Synthesis straight to 16-bit PCM: sub-bands ``[clips, channels * n_band, frames]`` -> int16 ``[clips, n_band * frames,
        channels]`` (interleaved WAV frames), ``clamp(round(inverse(x) * 32768), -32768, 32767)`` with the conversion and the
        interleave fused into the kernel's stores."""
        if x.dim() != 3:
            raise RuntimeError("inverse_pcm16 expects a 3-D tensor [batch, channels * n_band, frames]")
        return torch.ops.pqmf_b200.synthesis_pcm16(x, self.hk.float(), self._tables, self._inverse_delay(), self._flags)

    def _inverse_delay(self) -> int:
        return 0

    @torch.jit.export
    def inverse_bands(self, bands: List[torch.Tensor], n_frames: int, prev_tail: torch.Tensor, fade_out: torch.Tensor,
                      fade_in: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        """Per-band hand-off of the pitch-shifter pipeline (SURVEY 8f-3; reference ``1-PitchShifterWrapper.py:243-297``) as ONE call:
        ``bands`` are the ``n_band`` pitch-shifted sub-bands ``[B, len_k]`` (each of its own length); every band's first ``Lx`` samples
        are cross-faded with ``prev_tail[k]`` (``prev_tail * fade_out + band * fade_in``, batch 1 only, as in the reference), the band
        is centre-cropped / zero-padded to ``n_frames``, and the bands are synthesised -- all inside the kernel's loads, without the
        ``cat(dim=1)`` tensor.  Returns ``(signal [B, 1, n_band * n_frames], new prev_tail [n_band, Lx])``.  Pass an empty ``prev_tail``
        (``numel() == 0``) for no cross-fade."""
        return torch.ops.pqmf_b200.synthesis_bands(bands, self.hk.float(), n_frames, self._inverse_delay(), prev_tail, fade_out, fade_in, self._flags)

    @torch.jit.export
    def process(self, x: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        """``(inverse(forward(x)), forward(x))`` -- what the reference's ``PQMFWrapper.process`` computes (PQMFWrapper.py:81-92) --
        in one op (bit-identical to the two calls; the synthesis kernel walks its tiles last-to-first, so the tail of the
        sub-bands is read back from L2).  Under autograd it falls back to ``forward`` / ``inverse``."""
        if x.dim() != 3:
            raise RuntimeError("PQMF.process expects a 3-D tensor [batch, channels, time]")
        if self.n_band == 1:
            return x, x
        t = x.shape[-1]
        if self.polyphase and t % self.n_band != 0:
            raise RuntimeError("polyphase PQMF needs the number of samples to be a multiple of n_band")
        if torch.is_grad_enabled() and x.requires_grad:  # the fused op has no autograd kernel: same result through the two ops
            y = self.forward(x)
            return self.inverse(y), y
        return torch.ops.pqmf_b200.roundtrip(x, self.hk.float(), self._tables, t // self.n_band, 0, self._flags)


class _BankConv(nn.Module):
    """Weight holder standing in for the two ``cached_conv.Conv1d`` layers of the reference's CachedPQMF
    (pqmf.py:316-333): keeps the ``forward_conv.weight`` / ``inverse_conv.weight`` state_dict keys, the
    ``_pad`` / ``cumulative_delay`` attributes and ``script_cache()``.  The arithmetic itself runs in the
    fused kernels straight from ``hk``; these weights are not read on the hot path."""

    def __init__(self, weight: torch.Tensor, pad: int, stride: int, delay: int):
        super().__init__()
        self.weight = nn.Parameter(weight.clone(), requires_grad=False)
        self._pad = (pad, pad)
        self.stride = (stride,)
        self.cumulative_delay: int = delay

    def script_cache(self):
        pass


class CachedPQMF(PQMF):
    """Real-time variant (reference pqmf.py:306-354).

    Offline (default, what the reference's exported .ts files run): ``forward`` is the same function as
    ``PQMF.forward`` (also for T % n_band != 0, giving ceil(T / n_band) frames) and ``inverse`` is
    ``PQMF.inverse`` delayed by one frame.

    Streaming (``streaming=True`` or ``forward_stream`` / ``inverse_stream``): block-by-block processing with
    the FIR history carried in device-resident state, equal to one long causal run (SURVEY.md A.4):
    analysis is L/2 samples late, synthesis (K/2 + 1) frames late, ``cumulative_delay`` samples in total.
    """

    def __init__(self, *args, **kwargs):
        streaming = bool(kwargs.pop("streaming", False))
        super().__init__(*args, **kwargs)
        m, length = self.hk.shape
        k_taps = length // m if length % m == 0 else 0
        fwd_w = make_odd(self.hk).unsqueeze(1)
        self.forward_conv = _BankConv(fwd_w, fwd_w.shape[-1] // 2, m, 0)
        if k_taps:
            inv_w = make_odd(self.hk.flip(-1).reshape(m, k_taps, m).permute(2, 0, 1))
        else:  # non power-of-two classic bank: no polyphase synthesis weights exist in the reference either
            inv_w = torch.zeros(m, m, 1)
        self.inverse_conv = _BankConv(inv_w, inv_w.shape[-1] // 2, 1, 0)
        self.streaming: bool = streaming
        self.taps_per_phase: int = int(k_taps)
        self.cumulative_delay: int = int(length // 2 + (k_taps // 2) * m + m)
        self.register_buffer("_x_state", torch.zeros(2, 0, int(length)), persistent=False)
        self.register_buffer("_s_state", torch.zeros(2, 0, int(length)), persistent=False)
        self._x_slot: int = 0
        self._s_slot: int = 0
        self._frames_in: int = 0
        self._frames_out: int = 0

    def script_cache(self):
        self.forward_conv.script_cache()
        self.inverse_conv.script_cache()

    def _inverse_delay(self) -> int:
        return 1  # CachedPQMF.inverse is PQMF.inverse one frame later (pqmf.py:345-354)

    def _n_frames_of(self, t: int) -> int:
        return (t + self.n_band - 1) // self.n_band  # the cached analysis accepts ragged lengths: ceil(T / n_band) frames

    @torch.jit.export
    def reset_stream(self) -> None:
        """Forget all carried history (next block starts a new stream)."""
        self._x_state = torch.zeros(2, 0, self.hk.shape[1], device=self.hk.device)
        self._s_state = torch.zeros(2, 0, self.hk.shape[1], device=self.hk.device)
        self._x_slot = 0
        self._s_slot = 0
        self._frames_in = 0
        self._frames_out = 0

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        if x.dim() != 3:
            raise RuntimeError("CachedPQMF.forward expects a 3-D tensor [batch, channels, time]")
        if self.n_band == 1:
            return x
        if self.streaming:
            return self.forward_stream(x)
        n_frames = (x.shape[-1] + self.n_band - 1) // self.n_band
        return torch.ops.pqmf_b200.analysis(x, self.hk.float(), self._tables, n_frames, self._call_flags(x))

    @torch.jit.export
    def inverse(self, x: torch.Tensor) -> torch.Tensor:
        if x.dim() != 3:
            raise RuntimeError("CachedPQMF.inverse expects a 3-D tensor [batch, n_band, frames]")
        if self.n_band == 1:
            return x
        if self.streaming:
            return self.inverse_stream(x)
        return torch.ops.pqmf_b200.synthesis(x, self.hk.float(), self._tables, 1, self._call_flags(x))

    @torch.jit.export
    def process(self, x: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        """Offline ``(inverse(forward(x)), forward(x))`` in one op (see ``PQMF.process``); the reconstruction is one frame late,
        as ``CachedPQMF.inverse``."""
        if x.dim() != 3:
            raise RuntimeError("CachedPQMF.process expects a 3-D tensor [batch, channels, time]")
        if self.n_band == 1:
            return x, x
        if torch.is_grad_enabled() and x.requires_grad:
            y = self.forward(x)
            return self.inverse(y), y
        n_frames = (x.shape[-1] + self.n_band - 1) // self.n_band
        return torch.ops.pqmf_b200.roundtrip(x, self.hk.float(), self._tables, n_frames, 1, self._flags)

    @torch.jit.export
    def process_stream(self, x: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        """One streaming block step -- ``y = forward_stream(x); out = inverse_stream(y)`` -- as ONE op call (what ``PQMFWrapper.process``
        does per audio buffer; half the host-side dispatch of the two calls).  Returns ``(out, y)``; the same bits and the same state
        updates as the two calls."""
        rows = x.shape[0] * x.shape[1]
        length = self.hk.shape[1]
        if self._x_state.shape[1] != rows or self._x_state.device != x.device:
            self._x_state = torch.zeros(2, rows, length, device=x.device)
            self._x_slot = 0
            self._frames_in = 0
        if self._s_state.shape[1] != rows or self._s_state.device != x.device:
            self._s_state = torch.zeros(2, rows, length, device=x.device)
            self._s_slot = 0
            self._frames_out = 0
        out, y = torch.ops.pqmf_b200.stream_step(x, self.hk.float(), self._tables, self._x_state[self._x_slot], self._x_state[1 - self._x_slot],
                                                 self._s_state[self._s_slot], self._s_state[1 - self._s_slot], self._frames_in % 2,
                                                 self._frames_out % 2, self._flags)
        self._x_slot = 1 - self._x_slot
        self._s_slot = 1 - self._s_slot
        self._frames_in += x.shape[-1] // self.n_band
        self._frames_out += x.shape[-1] // self.n_band
        return out, y

    @torch.jit.export
    def process_stream_pcm16(self, pcm: torch.Tensor, downmix: bool = False) -> Tuple[torch.Tensor, torch.Tensor]:
        """``process_stream`` from 16-bit PCM to 16-bit PCM: ``pcm`` int16 ``[S, T_block, channels]`` (interleaved WAV frames) -> ``(pcm_out
        int16 [S, T_block, C'], y float32 [S, C' * n_band, T_block / n_band])`` with ``C' = 1`` when down-mixing, else ``channels``.  Bit-equal
        to ``process_stream`` on the widened block (``forward_pcm16``'s widening; row ``s * C' + c`` is channel ``c`` of block ``s``) followed by
        ``inverse_pcm16``'s quantisation, with the same state updates: PCM and float32 blocks continue one stream."""
        if pcm.dim() != 3:
            raise RuntimeError("process_stream_pcm16 expects int16 WAV frames [blocks, time, channels]")
        rows = pcm.shape[0] * (1 if downmix else pcm.shape[2])
        length = self.hk.shape[1]
        if self._x_state.shape[1] != rows or self._x_state.device != pcm.device:
            self._x_state = torch.zeros(2, rows, length, device=pcm.device)
            self._x_slot = 0
            self._frames_in = 0
        if self._s_state.shape[1] != rows or self._s_state.device != pcm.device:
            self._s_state = torch.zeros(2, rows, length, device=pcm.device)
            self._s_slot = 0
            self._frames_out = 0
        out, y = torch.ops.pqmf_b200.stream_step_pcm16(pcm, self.hk.float(), self._tables, self._x_state[self._x_slot],
                                                       self._x_state[1 - self._x_slot], self._s_state[self._s_slot], self._s_state[1 - self._s_slot],
                                                       self._frames_in % 2, self._frames_out % 2, downmix, self._flags)
        self._x_slot = 1 - self._x_slot
        self._s_slot = 1 - self._s_slot
        self._frames_in += pcm.shape[1] // self.n_band
        self._frames_out += pcm.shape[1] // self.n_band
        return out, y

    @torch.jit.export
    def forward_stream_pcm16(self, pcm: torch.Tensor, downmix: bool = False) -> torch.Tensor:
        """One block of streaming analysis from 16-bit PCM: int16 ``[S, T_block, channels]`` -> ``[S, C' * n_band, T_block / n_band]``,
        bit-equal to ``forward_stream`` on the widened block (see ``process_stream_pcm16``); updates the same state."""
        if pcm.dim() != 3:
            raise RuntimeError("forward_stream_pcm16 expects int16 WAV frames [blocks, time, channels]")
        rows = pcm.shape[0] * (1 if downmix else pcm.shape[2])
        length = self.hk.shape[1]
        if self._x_state.shape[1] != rows or self._x_state.device != pcm.device:
            self._x_state = torch.zeros(2, rows, length, device=pcm.device)
            self._x_slot = 0
            self._frames_in = 0
        y = torch.ops.pqmf_b200.analysis_stream_pcm16(pcm, self.hk.float(), self._tables, self._x_state[self._x_slot],
                                                      self._x_state[1 - self._x_slot], self._frames_in % 2, downmix, self._flags)
        self._x_slot = 1 - self._x_slot
        self._frames_in += pcm.shape[1] // self.n_band
        return y

    @torch.jit.export
    def inverse_stream_pcm16(self, s: torch.Tensor) -> torch.Tensor:
        """One block of streaming synthesis to 16-bit PCM: float32 ``[S, C * n_band, F_block]`` -> int16 ``[S, n_band * F_block, C]``,
        ``clamp(round(inverse_stream(s) * 32768), -32768, 32767)`` interleaved; updates the same state."""
        if s.dim() != 3:
            raise RuntimeError("inverse_stream_pcm16 expects a 3-D tensor [blocks, channels * n_band, frames]")
        rows = s.shape[0] * (s.shape[1] // self.n_band)
        length = self.hk.shape[1]
        if self._s_state.shape[1] != rows or self._s_state.device != s.device:
            self._s_state = torch.zeros(2, rows, length, device=s.device)
            self._s_slot = 0
            self._frames_out = 0
        out = torch.ops.pqmf_b200.synthesis_stream_pcm16(s, self.hk.float(), self._tables, self._s_state[self._s_slot],
                                                         self._s_state[1 - self._s_slot], self._frames_out % 2, self._flags)
        self._s_slot = 1 - self._s_slot
        self._frames_out += s.shape[-1]
        return out

    @torch.jit.export
    def forward_stream(self, x: torch.Tensor) -> torch.Tensor:
        """One block of streaming analysis: x [S, 1, T_block] -> [S, n_band, T_block / n_band]; updates state."""
        rows = x.shape[0] * x.shape[1]
        length = self.hk.shape[1]
        if self._x_state.shape[1] != rows or self._x_state.device != x.device:
            self._x_state = torch.zeros(2, rows, length, device=x.device)
            self._x_slot = 0
            self._frames_in = 0
        y = torch.ops.pqmf_b200.analysis_stream(x, self.hk.float(), self._tables, self._x_state[self._x_slot],
                                                self._x_state[1 - self._x_slot], self._frames_in % 2, self._flags)
        self._x_slot = 1 - self._x_slot
        self._frames_in += x.shape[-1] // self.n_band
        return y

    @torch.jit.export
    def inverse_stream(self, s: torch.Tensor) -> torch.Tensor:
        """One block of streaming synthesis: s [S, n_band, F_block] -> [S, 1, n_band * F_block]; updates state."""
        rows = s.shape[0] * (s.shape[1] // self.n_band)
        length = self.hk.shape[1]
        if self._s_state.shape[1] != rows or self._s_state.device != s.device:
            self._s_state = torch.zeros(2, rows, length, device=s.device)
            self._s_slot = 0
            self._frames_out = 0
        out = torch.ops.pqmf_b200.synthesis_stream(s, self.hk.float(), self._tables, self._s_state[self._s_slot],
                                                   self._s_state[1 - self._s_slot], self._frames_out % 2, self._flags)
        self._s_slot = 1 - self._s_slot
        self._frames_out += s.shape[-1]
        return out
