"""CUDA-graph replay of the real-time block step (forward_stream + inverse_stream of one block of every stream).

The reference's real-time use is one stream and blocks of 512 ... 16384 samples (PQMFWrapper.py:40-41: m_buffer_size / max_buffer_size,
driven block by block from a Pure Data external, README.md:16): there the two kernel launches take a few microseconds and the host
side of the call (op dispatch, output allocation, launch) dominates.  A captured graph removes it.  The streaming ops read their FIR
history from one buffer and write the new history to another (ping-pong), so a single graph would replay stale pointers; this helper
captures TWO graphs -- even and odd steps -- over fixed input / state / output buffers and alternates between them.

``StreamPool`` serves many independent sessions instead of one lockstep batch: each call steps any subset of the pool's streams, each
with its own history, ping-pong half and frame parity kept on the device.  A pool may take float32, float16 or bfloat16 blocks.
"""
from __future__ import annotations

import operator

from typing import List, Optional, Sequence, Tuple, Union

import torch


def _widen(pcm: torch.Tensor, downmix: bool) -> torch.Tensor:
    """int16 ``[S, T, C]`` -> float32 ``[S, C', T]`` with the PCM ops' arithmetic: v / 32768, the down-mix summed in channel order, then / C."""
    f = pcm.float().mul_(1.0 / 32768.0)
    if not downmix:
        return f.permute(0, 2, 1).contiguous()
    acc = f[..., 0].clone()
    for c in range(1, f.shape[-1]):
        acc.add_(f[..., c])
    return acc.div_(torch.full((), float(f.shape[-1]), device=acc.device)).unsqueeze(1)


# the names torch's C++ side gives dtypes in its errors ("x must be BFloat16 (the pool's dtype), got Float")
_ATEN_NAMES = {torch.float32: "Float", torch.float16: "Half", torch.bfloat16: "BFloat16", torch.float64: "Double", torch.int16: "Short",
               torch.int32: "Int", torch.int64: "Long"}
POOL_DTYPES = (torch.float32, torch.float16, torch.bfloat16)


def _check_dtype(t: torch.Tensor, dtype: torch.dtype, name: str) -> None:
    if t.dtype != dtype:
        raise RuntimeError(f"{name} must be {_ATEN_NAMES[dtype]} (the pool's dtype), got {_ATEN_NAMES.get(t.dtype, str(t.dtype))}")


def _quantise(v: torch.Tensor) -> torch.Tensor:
    """float32 ``[S, C, T]`` -> int16 ``[S, T, C]``: clamp(rint(v * 32768), -32768, 32767), the PCM ops' rounding."""
    return torch.clamp(torch.round(v * 32768.0), -32768.0, 32767.0).to(torch.int16).permute(0, 2, 1).contiguous()


class StreamGraph:
    """``g = StreamGraph(cached_pqmf, streams, block)``; then per block ``y, out = g.step(x_block)``.

    ``x_block`` ``[streams, 1, block]`` is copied into the graph's static input (or write into ``g.x`` yourself and call ``g.step()``);
    the returned sub-bands ``[streams, n_band, block / n_band]`` and signal ``[streams, 1, block]`` are the graph's static outputs
    of this step's parity: valid until the step after next.  ``block`` must hold an even number of frames (the sign mask follows the
    global frame parity, which a captured graph cannot advance)."""

    def __init__(self, mod, streams: int, block: int, device: Optional[torch.device] = None):
        if block % (2 * mod.n_band) != 0:
            raise ValueError(f"StreamGraph needs an even number of frames per block: block={block} is not a multiple of {2 * mod.n_band}")
        dev = torch.device(device) if device is not None else mod.hk.device
        if dev.type != "cuda":
            raise RuntimeError("StreamGraph needs the module on a CUDA device")
        self.mod = mod
        self.x = torch.zeros(streams, 1, block, device=dev)
        self._k = 0
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.no_grad(), torch.cuda.stream(side):
            mod.reset_stream()
            for _ in range(2):  # allocates the ping-pong state, opts the kernels into their shared memory: none of that may happen in a capture
                mod.process_stream(self.x)
            side.synchronize()
            assert mod._x_slot == 0 and mod._s_slot == 0
            self._graphs, self._outs = [], []
            for _ in range(2):
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=side):
                    out, y = mod.process_stream(self.x)
                self._graphs.append(g)
                self._outs.append((y, out))
        torch.cuda.current_stream(dev).wait_stream(side)
        self.reset()

    def reset(self) -> None:
        """Forget the carried history (zeroes the state buffers IN PLACE: the captured pointers stay valid)."""
        self.mod._x_state.zero_()
        self.mod._s_state.zero_()
        self._k = 0

    def step(self, x: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
        if x is not None:
            self.x.copy_(x, non_blocking=True)
        self._graphs[self._k & 1].replay()
        out = self._outs[self._k & 1]
        self._k += 1
        return out


class StreamPool:
    """Device-resident streaming state for ``capacity`` independent streams of one ``CachedPQMF``.

    ``pool = StreamPool(mod, capacity)``; then per call ``out, y = pool.step(x, ids)``: ``x`` ``[n, 1, T]`` holds the next block of each of
    the ``n`` distinct streams ``ids`` (in any order; streams not listed are left exactly as they are), and returns their signal
    ``[n, 1, T]`` and sub-bands ``[n, n_band, T / n_band]`` -- per row bit for bit what ``process_stream`` gives for that stream.
    ``forward`` / ``inverse`` run one direction, with its own state and parity as ``forward_stream`` / ``inverse_stream``; ``reset`` forgets
    streams so that a new session can take their slots.  ``step_pcm16`` / ``forward_pcm16`` / ``inverse_pcm16`` are the same calls with
    16-bit PCM blocks (interleaved WAV frames in, int16 samples out).  ``step_groups`` / ``forward_groups`` / ``inverse_groups`` take up
    to 8 groups of streams with their own block lengths in one call, ``step_groups_pcm16`` / ``forward_groups_pcm16`` /
    ``inverse_groups_pcm16`` the same with 16-bit PCM blocks.

    ``ids`` is a list of ints or a CPU integer tensor (checked: in range and distinct, else ``ValueError``), or a CUDA integer tensor, which
    is trusted as it is and costs no host synchronisation.  With CUDA ids a step allocates nothing but its outputs, so it can be captured
    in a CUDA graph: the frame parities live on the device, so one graph replays steps of one ``n`` and ``T`` for any ids and any
    number of frames per block.

    The pool reads ``mod.hk``, ``mod._tables`` and ``mod._flags`` at every call (``load_state_dict``, casts and ``refresh_tables`` carry
    through) and uses none of ``mod``'s own streaming state.  One pool is stepped from one CUDA stream at a time.

    ``dtype`` (float32, float16 or bfloat16; independent of the module's dtype) is the element type of the float blocks and sub-bands
    that ``step`` / ``forward`` / ``inverse`` and the grouped float calls take and return; a block of another dtype raises.  The pool's state
    stays float32 whatever the dtype.  On a half pool, per row ``forward(x)`` is bit for bit ``forward(x.float())`` of a float32 pool
    rounded to ``dtype``, ``inverse(y)`` likewise, and ``step(x)`` is ``forward`` followed by ``inverse`` of the ROUNDED sub-bands, with the
    state and phase words of that float32 pool.  ``step`` / ``forward`` / ``inverse`` and ``forward_groups`` / ``inverse_groups`` run the
    streaming Hankel-4 kernels with half loads and stores where the float32 pool would run those kernels; other calls are staged (widen,
    float32 call, round) direction by direction, and ``step_groups`` is ``forward_groups`` then ``inverse_groups``.  The PCM calls are those
    of a float32 pool."""

    def __init__(self, mod, capacity: int, dtype: torch.dtype = torch.float32):
        if capacity < 1:
            raise ValueError(f"StreamPool needs a capacity of at least 1, got {capacity}")
        if dtype not in POOL_DTYPES:
            raise ValueError(f"StreamPool dtype must be torch.float32, torch.float16 or torch.bfloat16, got {dtype}")
        dev = mod.hk.device
        if dev.type != "cuda":
            raise RuntimeError("StreamPool needs the module on a CUDA device")
        self.mod = mod
        self.capacity = int(capacity)
        self.dtype = dtype
        m, length = mod.hk.shape
        self.xpool = torch.zeros(2, capacity, length, device=dev)
        self.spool = torch.zeros(2, capacity, m, max(length // m, 1), device=dev)
        self.xphase = torch.zeros(capacity, dtype=torch.int32, device=dev)
        self.sphase = torch.zeros(capacity, dtype=torch.int32, device=dev)

    def _ids(self, ids: Union[torch.Tensor, Sequence[int]]) -> torch.Tensor:
        dev = self.xpool.device
        if isinstance(ids, torch.Tensor) and ids.is_cuda:
            if ids.dim() != 1 or ids.dtype.is_floating_point or ids.dtype.is_complex or ids.dtype == torch.bool:
                raise ValueError("ids must be a 1-D integer tensor")
            return ids.to(dev, torch.int32)
        if isinstance(ids, torch.Tensor) and (ids.dim() != 1 or ids.dtype.is_floating_point or ids.dtype == torch.bool):
            raise ValueError("ids must be a 1-D integer tensor")
        try:
            host = [operator.index(i) for i in (ids.tolist() if isinstance(ids, torch.Tensor) else ids)]
        except TypeError:
            raise ValueError("ids must be integers") from None
        bad = [i for i in host if not 0 <= i < self.capacity]
        if bad:
            raise ValueError(f"stream ids {bad[:8]} are outside the pool [0, {self.capacity})")
        if len(set(host)) != len(host):
            raise ValueError("stream ids must be distinct")
        return torch.tensor(host, dtype=torch.int32).to(dev)

    @property
    def _half(self) -> bool:
        return self.dtype != torch.float32

    def step(self, x: torch.Tensor, ids) -> Tuple[torch.Tensor, torch.Tensor]:
        """One block of the listed streams through analysis and synthesis: returns ``(out, y)``."""
        mod = self.mod
        if mod.n_band == 1:
            if self._half:
                _check_dtype(x, self.dtype, "x")
            return x, x
        if self._half:
            return torch.ops.pqmf_b200.stream_pool_step_x(x, mod.hk.float(), mod._tables, self.xpool, self.xphase, self.spool, self.sphase,
                                                          self._ids(ids), self.dtype, mod._flags)
        return torch.ops.pqmf_b200.stream_pool_step(x, mod.hk.float(), mod._tables, self.xpool, self.xphase, self.spool, self.sphase,
                                                    self._ids(ids), mod._flags)

    def forward(self, x: torch.Tensor, ids) -> torch.Tensor:
        """Streaming analysis of one block of the listed streams: ``[n, 1, T]`` -> ``[n, n_band, T / n_band]``."""
        mod = self.mod
        if mod.n_band == 1:
            if self._half:
                _check_dtype(x, self.dtype, "x")
            return x
        if self._half:
            return torch.ops.pqmf_b200.stream_pool_analysis_x(x, mod.hk.float(), mod._tables, self.xpool, self.xphase, self._ids(ids), self.dtype,
                                                              mod._flags)
        return torch.ops.pqmf_b200.stream_pool_analysis(x, mod.hk.float(), mod._tables, self.xpool, self.xphase, self._ids(ids), mod._flags)

    def inverse(self, y: torch.Tensor, ids) -> torch.Tensor:
        """Streaming synthesis of one block of the listed streams: ``[n, n_band, F]`` -> ``[n, 1, n_band * F]``."""
        mod = self.mod
        if mod.n_band == 1:
            if self._half:
                _check_dtype(y, self.dtype, "s")
            return y
        if self._half:
            return torch.ops.pqmf_b200.stream_pool_synthesis_x(y, mod.hk.float(), mod._tables, self.spool, self.sphase, self._ids(ids), self.dtype,
                                                               mod._flags)
        return torch.ops.pqmf_b200.stream_pool_synthesis(y, mod.hk.float(), mod._tables, self.spool, self.sphase, self._ids(ids), mod._flags)

    MAX_GROUPS = 8

    def _group_ids(self, groups) -> Tuple[List[torch.Tensor], List[torch.Tensor]]:
        """Blocks and ids of ``(block, ids)`` pairs; CPU ids are checked as in ``step``, and distinct across all groups."""
        groups = list(groups)
        if len(groups) > self.MAX_GROUPS:
            raise ValueError(f"at most {self.MAX_GROUPS} groups per call, got {len(groups)}")
        blocks, ids, seen = [], [], set()
        for block, gids in groups:
            t = self._ids(gids)
            if not (isinstance(gids, torch.Tensor) and gids.is_cuda):
                host = [operator.index(i) for i in (gids.tolist() if isinstance(gids, torch.Tensor) else gids)]
                if seen.intersection(host):
                    raise ValueError("stream ids must be distinct across all groups")
                seen.update(host)
            blocks.append(block)
            ids.append(t)
        return blocks, ids

    def step_groups(self, groups) -> List[Tuple[torch.Tensor, torch.Tensor]]:
        """``step`` of up to 8 groups ``(x_g [n_g, 1, T_g], ids_g)`` with their own block lengths, in one call: returns ``[(out_g, y_g)]``.

        The groups the streaming Hankel-4 kernels can take run together in one launch per direction when they make enough tiles together
        (so small groups of several block lengths reach the tensor cores); each of their rows is what those kernels give it in a pool
        call.  Every other group gives exactly what ``step(x_g, ids_g)`` gives; one group is ``step``.  ids follow ``step``'s rules and must
        be distinct across all groups.  On a half pool the call is ``forward_groups`` then ``inverse_groups`` of the rounded sub-bands: each
        direction joins the groups the float32 call of that direction would join."""
        if self._half:
            groups = list(groups)
            ys = self.forward_groups(groups)
            outs = self.inverse_groups([(y, gids) for y, (_, gids) in zip(ys, groups)])
            return list(zip(outs, ys))
        blocks, ids = self._group_ids(groups)
        mod = self.mod
        if mod.n_band == 1:
            return [(x, x) for x in blocks]
        outs, ys = torch.ops.pqmf_b200.stream_pool_step_groups(blocks, mod.hk.float(), mod._tables, self.xpool, self.xphase, self.spool,
                                                               self.sphase, ids, mod._flags)
        return list(zip(outs, ys))

    def forward_groups(self, groups) -> List[torch.Tensor]:
        """``forward`` of up to 8 groups ``(x_g [n_g, 1, T_g], ids_g)`` in one call (routed as ``step_groups``): returns ``[y_g]``.  On a
        half pool per row the float32 call on the widened blocks, rounded; the joined groups run one half-precision launch."""
        blocks, ids = self._group_ids(groups)
        mod = self.mod
        if self._half:
            for b in blocks:
                _check_dtype(b, self.dtype, "x")
        if mod.n_band == 1:
            return [b.float().to(self.dtype) for b in blocks] if self._half else blocks
        if self._half:
            return list(torch.ops.pqmf_b200.stream_pool_analysis_groups_x(blocks, mod.hk.float(), mod._tables, self.xpool, self.xphase, ids,
                                                                          self.dtype, mod._flags))
        return list(torch.ops.pqmf_b200.stream_pool_analysis_groups(blocks, mod.hk.float(), mod._tables, self.xpool, self.xphase, ids, mod._flags))

    def inverse_groups(self, groups) -> List[torch.Tensor]:
        """``inverse`` of up to 8 groups ``(y_g [n_g, n_band, F_g], ids_g)`` in one call (routed as ``step_groups``): returns ``[out_g]``.  On
        a half pool per row the float32 call on the widened sub-bands, rounded; the joined groups run one half-precision launch."""
        blocks, ids = self._group_ids(groups)
        mod = self.mod
        if self._half:
            for b in blocks:
                _check_dtype(b, self.dtype, "s")
        if mod.n_band == 1:
            return [b.float().to(self.dtype) for b in blocks] if self._half else blocks
        if self._half:
            return list(torch.ops.pqmf_b200.stream_pool_synthesis_groups_x(blocks, mod.hk.float(), mod._tables, self.spool, self.sphase, ids,
                                                                           self.dtype, mod._flags))
        return list(torch.ops.pqmf_b200.stream_pool_synthesis_groups(blocks, mod.hk.float(), mod._tables, self.spool, self.sphase, ids, mod._flags))

    def step_pcm16(self, pcm: torch.Tensor, ids, downmix: bool = False) -> Tuple[torch.Tensor, torch.Tensor]:
        """``step`` from 16-bit PCM to 16-bit PCM: ``pcm`` int16 ``[S, T, channels]`` -> ``(pcm_out int16 [S, T, C'], y [S, C' * n_band,
        T / n_band])``, ``C' = 1`` when down-mixing, else ``channels``.  ``ids`` has one stream per row: row ``r * C' + c`` (channel ``c`` of
        block ``r``) is stream ``ids[r * C' + c]``.  Per row bit-equal to ``step`` on the widened block (``CachedPQMF.forward_pcm16``'s
        widening), then quantised (``inverse_pcm16``'s rounding); the same pool and phase-word updates."""
        mod = self.mod
        return torch.ops.pqmf_b200.stream_pool_step_pcm16(pcm, mod.hk.float(), mod._tables, self.xpool, self.xphase, self.spool, self.sphase,
                                                          self._ids(ids), downmix, mod._flags)

    def forward_pcm16(self, pcm: torch.Tensor, ids, downmix: bool = False) -> torch.Tensor:
        """``forward`` from 16-bit PCM: int16 ``[S, T, channels]`` -> ``[S, C' * n_band, T / n_band]`` (rows and ids as ``step_pcm16``)."""
        mod = self.mod
        return torch.ops.pqmf_b200.stream_pool_analysis_pcm16(pcm, mod.hk.float(), mod._tables, self.xpool, self.xphase, self._ids(ids), downmix,
                                                              mod._flags)

    def inverse_pcm16(self, s: torch.Tensor, ids) -> torch.Tensor:
        """``inverse`` to 16-bit PCM: ``[S, C * n_band, F]`` -> int16 ``[S, n_band * F, C]``; row ``r * C + c`` is stream ``ids[r * C + c]``."""
        mod = self.mod
        return torch.ops.pqmf_b200.stream_pool_synthesis_pcm16(s, mod.hk.float(), mod._tables, self.spool, self.sphase, self._ids(ids), mod._flags)

    def step_groups_pcm16(self, groups, downmix: bool = False) -> List[Tuple[torch.Tensor, torch.Tensor]]:
        """``step_pcm16`` of up to 8 groups ``(pcm_g int16 [S_g, T_g, C_g], ids_g)`` with their own block lengths and channel counts, in one
        call: returns ``[(pcm_out_g int16 [S_g, T_g, C'_g], y_g [S_g, C'_g * n_band, T_g / n_band])]``; ``downmix`` applies to every group.

        Rows and ids of a group follow ``step_pcm16``; ids follow ``step_groups`` (distinct across all groups).  Per row bit-equal to
        ``step_groups`` on the widened blocks, then quantised, with the same pool and phase-word updates: the groups ``step_groups`` would
        run together run together here, with PCM loads and stores in the kernels.  One group is ``step_pcm16``."""
        blocks, ids = self._group_ids(groups)
        mod = self.mod
        if mod.n_band == 1:
            return [(_quantise(w), w) for w in (_widen(b, downmix) for b in blocks)]
        outs, ys = torch.ops.pqmf_b200.stream_pool_step_groups_pcm16(blocks, mod.hk.float(), mod._tables, self.xpool, self.xphase, self.spool,
                                                                     self.sphase, ids, downmix, mod._flags)
        return list(zip(outs, ys))

    def forward_groups_pcm16(self, groups, downmix: bool = False) -> List[torch.Tensor]:
        """``forward_pcm16`` of up to 8 groups ``(pcm_g int16 [S_g, T_g, C_g], ids_g)`` in one call (routed as ``step_groups_pcm16``):
        returns ``[y_g [S_g, C'_g * n_band, T_g / n_band]]``."""
        blocks, ids = self._group_ids(groups)
        mod = self.mod
        if mod.n_band == 1:
            return [_widen(b, downmix) for b in blocks]
        return list(torch.ops.pqmf_b200.stream_pool_analysis_groups_pcm16(blocks, mod.hk.float(), mod._tables, self.xpool, self.xphase, ids,
                                                                          downmix, mod._flags))

    def inverse_groups_pcm16(self, groups) -> List[torch.Tensor]:
        """``inverse_pcm16`` of up to 8 groups ``(s_g [S_g, C_g * n_band, F_g], ids_g)`` in one call (routed as ``step_groups_pcm16``):
        returns ``[pcm_out_g int16 [S_g, n_band * F_g, C_g]]``; row ``r * C_g + c`` of a group is stream ``ids_g[r * C_g + c]``."""
        blocks, ids = self._group_ids(groups)
        mod = self.mod
        if mod.n_band == 1:
            return [_quantise(s) for s in blocks]
        return list(torch.ops.pqmf_b200.stream_pool_synthesis_groups_pcm16(blocks, mod.hk.float(), mod._tables, self.spool, self.sphase, ids,
                                                                           mod._flags))

    def reset(self, ids=None) -> None:
        """Forget the listed streams (all when ``ids`` is None): zero history in both directions, parity 0; in place, on the device."""
        if ids is None:
            for t in (self.xpool, self.spool, self.xphase, self.sphase):
                t.zero_()
            return
        idx = self._ids(ids).long()
        self.xpool.index_fill_(1, idx, 0.0)
        self.spool.index_fill_(1, idx, 0.0)
        self.xphase.index_fill_(0, idx, 0)
        self.sphase.index_fill_(0, idx, 0)
