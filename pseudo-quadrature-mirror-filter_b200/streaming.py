"""CUDA-graph replay of the real-time block step (forward_stream + inverse_stream of one block of every stream).

The reference's real-time use is one stream and blocks of 512 ... 16384 samples (PQMFWrapper.py:40-41: m_buffer_size / max_buffer_size,
driven block by block from a Pure Data external, README.md:16): there the two kernel launches take a few microseconds and the host
side of the call (op dispatch, output allocation, launch) dominates.  A captured graph removes it.  The streaming ops read their FIR
history from one buffer and write the new history to another (ping-pong), so a single graph would replay stale pointers; this helper
captures TWO graphs -- even and odd steps -- over fixed input / state / output buffers and alternates between them.

``StreamPool`` serves many independent sessions instead of one lockstep batch: each call steps any subset of the pool's streams, each
with its own history, ping-pong half and frame parity kept on the device.
"""
from __future__ import annotations

import operator

from typing import Optional, Sequence, Tuple, Union

import torch


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
    """Device-resident streaming state for ``capacity`` independent streams of one ``CachedPQMF`` (fp32).

    ``pool = StreamPool(mod, capacity)``; then per call ``out, y = pool.step(x, ids)``: ``x`` ``[n, 1, T]`` holds the next block of each of
    the ``n`` distinct streams ``ids`` (in any order; streams not listed are left exactly as they are), and returns their signal
    ``[n, 1, T]`` and sub-bands ``[n, n_band, T / n_band]`` -- per row bit for bit what ``process_stream`` gives for that stream.
    ``forward`` / ``inverse`` run one direction, with its own state and parity as ``forward_stream`` / ``inverse_stream``; ``reset`` forgets
    streams so that a new session can take their slots.

    ``ids`` is a list of ints or a CPU integer tensor (checked: in range and distinct, else ``ValueError``), or a CUDA integer tensor, which
    is trusted as it is and costs no host synchronisation.  With CUDA ids a step allocates nothing but its outputs, so it can be captured
    in a CUDA graph: the frame parities live on the device, so one graph replays steps of one ``n`` and ``T`` for any ids and any
    number of frames per block.

    The pool reads ``mod.hk``, ``mod._tables`` and ``mod._flags`` at every call (``load_state_dict``, casts and ``refresh_tables`` carry
    through) and uses none of ``mod``'s own streaming state.  One pool is stepped from one CUDA stream at a time."""

    def __init__(self, mod, capacity: int):
        if capacity < 1:
            raise ValueError(f"StreamPool needs a capacity of at least 1, got {capacity}")
        dev = mod.hk.device
        if dev.type != "cuda":
            raise RuntimeError("StreamPool needs the module on a CUDA device")
        self.mod = mod
        self.capacity = int(capacity)
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

    def step(self, x: torch.Tensor, ids) -> Tuple[torch.Tensor, torch.Tensor]:
        """One block of the listed streams through analysis and synthesis: returns ``(out, y)``."""
        mod = self.mod
        if mod.n_band == 1:
            return x, x
        return torch.ops.pqmf_b200.stream_pool_step(x, mod.hk.float(), mod._tables, self.xpool, self.xphase, self.spool, self.sphase,
                                                    self._ids(ids), mod._flags)

    def forward(self, x: torch.Tensor, ids) -> torch.Tensor:
        """Streaming analysis of one block of the listed streams: ``[n, 1, T]`` -> ``[n, n_band, T / n_band]``."""
        mod = self.mod
        if mod.n_band == 1:
            return x
        return torch.ops.pqmf_b200.stream_pool_analysis(x, mod.hk.float(), mod._tables, self.xpool, self.xphase, self._ids(ids), mod._flags)

    def inverse(self, y: torch.Tensor, ids) -> torch.Tensor:
        """Streaming synthesis of one block of the listed streams: ``[n, n_band, F]`` -> ``[n, 1, n_band * F]``."""
        mod = self.mod
        if mod.n_band == 1:
            return y
        return torch.ops.pqmf_b200.stream_pool_synthesis(y, mod.hk.float(), mod._tables, self.spool, self.sphase, self._ids(ids), mod._flags)

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
