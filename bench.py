#!/usr/bin/env python
"""Benchmark of the PQMF hot path (BASELINE.json metric: PQMF analyze+inverse Msamples/s, n_band=16).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one process per GPU under torchrun)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU algorithm (oracle port) on the host cores
    python bench.py --steps K --dump-outputs DIR            # also writes what the last timed step computed to DIR/*.npy

A "step" is one pass of the hot path -- PQMF.forward then PQMF.inverse -- over one batch of synthetic audio.
Workload = BASELINE.json configs[1]: 64 x 2^20 mono samples per GPU, n_band 16, attenuation 100, polyphase.
  value     : whole-job Msamples/s with inputs resident in HBM (device-timed with CUDA events, max over ranks)
  e2e       : the same metric through the C ABI host entry point (pinned HOST buffers in and out, copies in the timed region)
  roofline  : dominant kernel's algorithmic HBM bytes / its event-timed duration, against MEASURED_PEAKS.json
  cpu_baseline : the oracle's torch-CPU port of the reference algorithm on a bounded sample (rank 0, N=1 only)
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark may run from a read-only checkout: it leaves nothing in the tree

METRIC = "PQMF analyze+inverse throughput (n_band=16)"
UNIT = "Msamples/s"
BATCH, N_SAMPLES, N_BAND, ATTEN = 64, 1 << 20, 16, 100
WORKLOAD = "configs[1]: batch 64 x 2^20-sample synthetic mono, n_band=16 attenuation=100 polyphase forward+inverse per GPU"
ALGO_BYTES_PER_SAMPLE_PER_DIRECTION = 8  # 4 B read + 4 B written, sub-bands materialised (SURVEY.md 8d)


def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


def recorded_traffic():
    """dram bytes per launch of the dominant kernel from the committed `ncu --set full` capture, if any."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        with open(path) as f:
            return json.load(f)
    except Exception:
        return {}


class ClockSampler(threading.Thread):
    """Polls NVML for SM clock / throttle reasons while the timed region runs."""

    def __init__(self, index: int, period_s: float = 0.004):
        super().__init__(daemon=True)
        self.index, self.period, self.samples, self.reasons, self.max_mhz = index, period_s, [], set(), None
        self.power_w = []
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.nv = None

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._halt.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    self.power_w.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
                except Exception:
                    pass
                try:
                    mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def sample_now(self):
        """One sample taken by the caller (used while the GPU is still working through the queued steps, so that even a very
        short timed region has at least one sample under load)."""
        if not self.ok:
            return
        try:
            self.samples.append(int(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
            self.power_w.append(self.nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
            mask = int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            for bit, name in ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap")):
                if mask & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def stop(self):
        self._halt.set()
        self.join(timeout=1.0)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s), "power_w_max": (round(max(self.power_w), 1) if self.power_w else None)}


def physical_gpu_index(local_rank: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


# ----------------------------------------------------------------------------------------------------------------
def cpu_port_throughput(batch: int, n_samples: int, repeats: int, warmup: int):
    """Oracle port (torch CPU, all host threads) of the reference algorithm: Msamples/s of forward+inverse."""
    import torch

    from oracle import pqmf_oracle as O
    from oracle import pqmf_port_torch as P

    _, hk = O.design_bank(ATTEN, N_BAND)
    f, i, threads = P.time_roundtrip(torch.from_numpy(hk), batch, n_samples, repeats=repeats, warmup=warmup)
    return batch * n_samples / (f + i) * 1e-6, threads, f, i


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    # the SAME workload as the GPU arm: all 64 rows of 2^20 samples per step (~0.3 s of host work per step on the GPU box's 16
    # threads), the same warm-up count; the step count is bounded so that the run ends within a few minutes on any host
    batch = BATCH
    steps, warmup = max(1, min(args.steps, 30)), max(1, min(args.warmup, 5))
    val, threads, f, i = cpu_port_throughput(batch, N_SAMPLES, repeats=steps, warmup=warmup)
    sample = (f"{batch} x 2^20 samples per step (the whole configs[1] batch), best of {steps} steps after {warmup} warm-up; torch-CPU port of "
              f"pqmf.py:115-157 on {threads} threads")
    line = {
        "impl": "reference", "metric": METRIC, "value": round(val, 3), "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
        "ms_per_step": round((f + i) * 1e3, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": WORKLOAD, "n_band": N_BAND, "batch_per_gpu": BATCH, "samples_per_row": N_SAMPLES,
                   "timing": "host wall clock (time.perf_counter)"},
        "cpu_baseline": {"value": round(val, 3), "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": round(val, 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ----------------------------------------------------------------------------------------------------------------
def run_gpu(args):
    import torch
    import torch.distributed as dist

    import pqmf_b200 as pq
    from pqmf_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (pqmf_b200 has no CPU path); use --impl reference for the CPU baseline")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    distributed = world > 1
    if distributed:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    n_gpus = world if distributed else 1
    steps, warmup = args.steps, max(3, args.warmup)

    # rows are independent: each rank owns its own 64 x 2^20 shard (weak scaling), no collective on the data path
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    x = (0.5 * torch.randn(BATCH, 1, N_SAMPLES, device=dev, generator=gen)).clamp_(-1.0, 1.0)
    mod = pq.PQMF(ATTEN, N_BAND).to(dev)
    stream = torch.cuda.current_stream()

    def step():
        y = mod(x)
        return y, mod.inverse(y)

    for _ in range(warmup):
        y, out = step()
    torch.cuda.synchronize()
    # parity guard inside the benchmark: near-perfect reconstruction of the interior (SURVEY section 6: ~60 dB on noise)
    err = (out[..., 4096:-4096] - x[..., 4096:-4096]).double()
    snr_db = float(10 * torch.log10((x[..., 4096:-4096].double() ** 2).sum() / (err ** 2).sum()))
    assert snr_db > 55.0, f"round-trip SNR {snr_db:.1f} dB: the kernels are not computing the PQMF"

    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
    sampler = ClockSampler(physical_gpu_index(local_rank))
    launches0 = pq.launch_count()
    if distributed:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.start()
    for k in range(steps):
        ev[k][0].record(stream)
        y = mod(x)
        ev[k][1].record(stream)
        out = mod.inverse(y)
        ev[k][2].record(stream)
    sampler.sample_now()  # the launches above only queue work: the GPU is still inside the timed region here
    torch.cuda.synchronize()
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, y, out)
    if distributed:
        dist.barrier()
    launches = pq.launch_count() - launches0
    total_ms = ev[0][0].elapsed_time(ev[-1][2])
    t_an = sum(e[0].elapsed_time(e[1]) for e in ev) / steps
    t_sy = sum(e[1].elapsed_time(e[2]) for e in ev) / steps
    if distributed:
        t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    ms_per_step = total_ms / steps
    value = n_gpus * BATCH * N_SAMPLES / (ms_per_step * 1e-3) * 1e-6

    # ---- end to end through the C ABI host entry point: pinned host buffers, H2D + kernels + D2H inside the timed region
    e2e_steps = max(2, min(steps, 10))
    hx = torch.empty(BATCH, N_SAMPLES, dtype=torch.float32).pin_memory()
    ho = torch.empty(BATCH, N_SAMPLES, dtype=torch.float32).pin_memory()
    hx.copy_(x[:, 0].cpu())
    hk_h = mod.hk.cpu().contiguous()
    tab_h = mod._tables.cpu().contiguous()
    flags = int(mod._flags)

    def host_step():
        rc = _lib.cabi.pqmf_roundtrip_host_f32(hx.data_ptr(), None, ho.data_ptr(), hk_h.data_ptr(), tab_h.data_ptr() if tab_h.numel() else None,
                                               BATCH, N_SAMPLES, N_BAND, int(hk_h.shape[1]), 0, flags, local_rank)
        _lib.check(rc, "pqmf_roundtrip_host_f32")

    for _ in range(2):
        host_step()
    assert torch.allclose(ho[:4, 5000:6000], out[:4, 0, 5000:6000].cpu(), atol=1e-6), "host entry point disagrees with the module path"
    if distributed:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        host_step()  # synchronises internally before returning
    e2e_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
    if distributed:
        t = torch.tensor([e2e_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    e2e_value = n_gpus * BATCH * N_SAMPLES / (e2e_ms * 1e-3) * 1e-6

    # ---- the same end to end with 16-bit PCM on both sides of the link (SURVEY 8f-4: the reference's inputs are int16 WAVs): the
    #      conversion happens inside the kernels' loads / stores, so 2 B/sample cross PCIe each way instead of 4.  A SECOND number,
    #      reported beside the fp32 headline, never instead of it.
    hp = (x[:, 0] * 32767.0).round().to(torch.int16).cpu().reshape(BATCH, N_SAMPLES, 1).pin_memory()
    hop = torch.empty_like(hp).pin_memory()

    def host_step_pcm():
        rc = _lib.cabi.pqmf_roundtrip_host_pcm16(hp.data_ptr(), None, hop.data_ptr(), hk_h.data_ptr(), tab_h.data_ptr() if tab_h.numel() else None,
                                                 BATCH, N_SAMPLES, 1, N_BAND, int(hk_h.shape[1]), 0, flags, local_rank)
        _lib.check(rc, "pqmf_roundtrip_host_pcm16")

    for _ in range(2):
        host_step_pcm()
    # near-perfect reconstruction survives the 16-bit quantisation: the output frames sit within a few LSB of the input frames
    pcm_err = (hop[:4, 4096:-4096, 0].to(torch.int32) - hp[:4, 4096:-4096, 0].to(torch.int32)).abs().float().mean().item()
    assert pcm_err < 40.0, f"PCM round trip is off by {pcm_err:.1f} LSB on average"
    if distributed:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        host_step_pcm()
    pcm_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
    pcm_ms = _max_over_ranks(torch, dist, dev, pcm_ms, distributed)
    pcm_value = n_gpus * BATCH * N_SAMPLES / (pcm_ms * 1e-3) * 1e-6
    _lib.cabi.pqmf_host_release()
    del hx, ho, hp, hop

    peak, peak_src = measured_peak_gbs()
    other = None if args.no_other_configs else other_configs(torch, dist, pq, dev, mod, x, peak, n_gpus, distributed)

    if rank != 0:
        if distributed:
            dist.destroy_process_group()
        return 0

    algo_bytes = ALGO_BYTES_PER_SAMPLE_PER_DIRECTION * BATCH * N_SAMPLES
    kernels = {
        "h4_analysis_kernel": {"ms": t_an, "gbs": algo_bytes / (t_an * 1e-3) * 1e-9},
        "h4_synthesis_kernel": {"ms": t_sy, "gbs": algo_bytes / (t_sy * 1e-3) * 1e-9},
    }
    dominant = max(kernels, key=lambda k: kernels[k]["ms"])
    traffic = recorded_traffic().get(dominant)  # NOT measured in this run: ncu counters cannot be read while timing
    roofline = {
        "bound": "hbm", "kernel": dominant, "achieved": round(kernels[dominant]["gbs"], 1), "peak": peak, "unit": "GB/s",
        "frac": round(kernels[dominant]["gbs"] / peak, 4), "traffic": traffic,
        "traffic_source": "profiles/traffic.json: dram__bytes_read.sum + dram__bytes_write.sum of one launch of this kernel from the committed ncu --set full capture",
        "peak_source": peak_src,
        "algorithmic_bytes_per_launch": algo_bytes,
        "per_kernel": {k: {"ms": round(v["ms"], 4), "achieved_gbs": round(v["gbs"], 1), "frac": round(v["gbs"] / peak, 4)} for k, v in kernels.items()},
        "round_trip_frac": round(2 * algo_bytes / ((t_an + t_sy) * 1e-3) * 1e-9 / peak, 4),
    }
    # ---- informational: the same kernels outside the power-capped steady state, and the other BASELINE configs (not the metric)
    cpu = None
    if n_gpus == 1 and not args.no_cpu_baseline:
        cb, cr = 8, 5
        cval, threads, f, i = cpu_port_throughput(cb, N_SAMPLES, repeats=cr, warmup=2)
        cpu = {"value": round(cval, 3), "unit": UNIT, "cores": threads, "kind": "port",
               "sample": f"{cb} x 2^20 samples (1/8 of the batch), best of {cr} after 2 warm-ups, torch-CPU port of the reference's conv1d path "
                         f"(forward {f*1e3:.1f} ms + inverse {i*1e3:.1f} ms)"}
    line = {
        "metric": METRIC, "value": round(value, 1), "unit": UNIT, "n_gpus": n_gpus, "steps": steps, "warmup": warmup,
        "ms_per_step": round(ms_per_step, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": WORKLOAD, "n_band": N_BAND, "batch_per_gpu": BATCH, "samples_per_row": N_SAMPLES, "sharding": f"rows x{n_gpus}, no collective",
                   "l2": "per-step working set 805 MB per GPU (x, sub-bands, out) exceeds the 126 MB L2; no flush needed",
                   "round_trip_snr_db": round(snr_db, 2)},
        "clocks": clocks,
        "e2e": {"value": round(e2e_value, 1), "unit": UNIT, "h2d_bytes_per_step": n_gpus * BATCH * N_SAMPLES * 4, "d2h_bytes_per_step": n_gpus * BATCH * N_SAMPLES * 4,
                "ms_per_step": round(e2e_ms, 3), "steps": e2e_steps, "api": "pqmf_roundtrip_host_f32 (C ABI, pinned host buffers, 8 MiB row chunks, 4 in flight, copy and kernel streams)"},
        "e2e_pcm16": {"value": round(pcm_value, 1), "unit": UNIT, "h2d_bytes_per_step": n_gpus * BATCH * N_SAMPLES * 2, "d2h_bytes_per_step": n_gpus * BATCH * N_SAMPLES * 2,
                      "ms_per_step": round(pcm_ms, 3), "steps": e2e_steps, "api": "pqmf_roundtrip_host_pcm16 (int16 WAV frames in pinned host memory in and out; "
                      "second number beside the fp32 headline)"},
        "gpu_launches": int(launches),
        "roofline": roofline,
        "cpu_baseline": cpu,
        "other_configs": other,
    }
    print(json.dumps(line))
    if distributed:
        dist.destroy_process_group()
    return 0


DUMP_ROWS = 4  # whole rows of the batch: sub-bands + reconstruction of 4 rows are 32 MiB, inside the 64 MB a dump may take


def dump_outputs(dirname: str, y, out):
    """Writes what the timed step returns to its caller -- the sub-bands of PQMF.forward [rows, 16, 65536] and the reconstruction of
    PQMF.inverse [rows, 1, 2^20] -- for a fixed, seeded sample of DUMP_ROWS rows (the same rows on every run) as float32 .npy files, so
    that two builds run with the same arguments can be compared output for output."""
    import numpy as np
    import torch

    rows = np.sort(np.random.default_rng(0).choice(BATCH, DUMP_ROWS, replace=False))
    idx = torch.from_numpy(rows).to(y.device)
    os.makedirs(dirname, exist_ok=True)
    for name, t in (("subbands", y), ("reconstruction", out)):
        np.save(os.path.join(dirname, f"{name}.npy"), t.index_select(0, idx).to(torch.float32).cpu().numpy())


def _max_over_ranks(torch, dist, dev, ms: float, distributed: bool) -> float:
    if not distributed:
        return ms
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def _sustained(torch, fn, seconds: float, min_steps: int = 10, max_steps: int = 2000):
    """ms per call of `fn` over a back-to-back run of about `seconds` (CUDA events on the current stream; the step count is fixed
    from a short calibration so that every rank times the same number of steps)."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        fn()
    e1.record()
    torch.cuda.synchronize()
    est = max(e0.elapsed_time(e1) / 3, 1e-3)
    steps = int(min(max_steps, max(min_steps, seconds * 1e3 / est)))
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps, steps


def _burst(torch, fn, n=5, inner=6):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    best = float("inf")
    for _ in range(n):
        fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(inner):
            fn()
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) / inner)
    return best


def bench_config3(torch, pq, dev, seconds):
    """configs[2]: 4096 concurrent streams x block 2048, state carried across blocks (CachedPQMF streaming mode), per GPU.
    One step = forward_stream + inverse_stream of one block of every stream.  Algorithmic bytes: 16 B/sample + the 8192 B of
    state traffic per stream-block of the explicit-state formulation = 20 B/sample (SURVEY 8d)."""
    streams, block = 4096, 2048
    gen = torch.Generator(device=dev).manual_seed(33)
    xs = (0.5 * torch.randn(streams, 1, block, device=dev, generator=gen)).clamp_(-1, 1)
    cached = pq.CachedPQMF(ATTEN, N_BAND).to(dev)

    def step():
        cached.process_stream(xs)   # forward_stream + inverse_stream as one op call

    ms, steps = _sustained(torch, step, seconds, min_steps=64)
    return {"workload": "configs[2]: 4096 streams x block 2048 per GPU, state carried", "samples_per_step": streams * block, "steps": steps, "ms": ms,
            "bytes_per_sample": 20}


def bench_config4(torch, pq, dev, seconds):
    """configs[3]: n_band 4 / 8 / 32 / 64 on 8-channel 48 kHz 60 s clips folded into the batch (8 clips -> 64 rows x 2 880 000), per GPU."""
    rows, t = 64, 2_880_000
    gen = torch.Generator(device=dev).manual_seed(44)
    x = (0.5 * torch.randn(rows, 1, t, device=dev, generator=gen)).clamp_(-1, 1)
    out = {}
    for m in (4, 8, 32, 64):
        bank = pq.PQMF(ATTEN, m).to(dev)
        y = bank(x)
        ta, _ = _sustained(torch, lambda: bank(x), seconds / 8, min_steps=5)
        ts, _ = _sustained(torch, lambda: bank.inverse(y), seconds / 8, min_steps=5)
        out[m] = (ta, ts)
        del y, bank
    return {"workload": "configs[3]: 8 clips x 8 ch x 60 s @ 48 kHz folded to 64 rows x 2 880 000 per GPU, n_band 4/8/32/64 (polyphase; classic runs the same kernel)",
            "samples_per_step": rows * t, "per_band_ms": out, "bytes_per_sample": 16}


def bench_config5(torch, pq, dev, seconds):
    """configs[4]: one GPU's shard of 8192 stereo clips x 10 s @ 48 kHz = 2048 rows x 480 000, CachedPQMF.forward + .inverse."""
    rows, t = 2048, 480_000
    x = torch.empty(rows, 1, t, device=dev)
    x.normal_(0, 0.5).clamp_(-1, 1)
    mod = pq.CachedPQMF(ATTEN, N_BAND).to(dev)
    holder = {}

    def step():
        holder["y"] = mod(x)
        holder["o"] = mod.inverse(holder["y"])

    ms, steps = _sustained(torch, step, seconds, min_steps=5, max_steps=200)
    return {"workload": "configs[4]: 2048 rows x 480 000 samples per GPU (8192 stereo clips x 10 s @ 48 kHz over 8 GPUs), CachedPQMF forward+inverse",
            "samples_per_step": rows * t, "steps": steps, "ms": ms, "bytes_per_sample": 16}


def bench_single_stream_latency(torch, pq, dev):
    """The reference's real-time use (PQMFWrapper.py:40-41: one stream, host blocks of 512 ... 16384 samples): microseconds per block
    step (process_stream = forward_stream + inverse_stream, state carried) -- eager module calls, wall clock including the host side of every call,
    and CUDA-graph replay (pq.StreamGraph) -- next to the real-time budget of the block at 44.1 kHz."""
    out = {}
    for block in (512, 2048, 8192, 16384):
        mod = pq.CachedPQMF(ATTEN, N_BAND).to(dev)
        xb = (0.5 * torch.randn(1, 1, block, device=dev)).clamp_(-1, 1)
        n = 200
        with torch.no_grad():
            for _ in range(10):
                mod.process_stream(xb)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(n):
                mod.process_stream(xb)
            torch.cuda.synchronize()
            eager_us = (time.perf_counter() - t0) / n * 1e6
            g = pq.StreamGraph(pq.CachedPQMF(ATTEN, N_BAND).to(dev), 1, block)
            for _ in range(10):
                g.step()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(n):
                g.step()
            torch.cuda.synchronize()
            graph_us = (time.perf_counter() - t0) / n * 1e6
            # one isolated step, host call to results visible on the host: the latency a real-time caller sees
            lat = []
            for _ in range(20):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                g.step()
                torch.cuda.synchronize()
                lat.append((time.perf_counter() - t0) * 1e6)
            lat.sort()
        out[f"block{block}"] = {"eager_us_per_step": round(eager_us, 1), "graph_us_per_step": round(graph_us, 1), "graph_isolated_step_us_median": round(lat[len(lat) // 2], 1),
                                "realtime_budget_us_at_44k1": round(block / 44100 * 1e6, 1)}
    return out


def other_configs(torch, dist, pq, dev, mod, x, peak, n_gpus, distributed):
    """The other BASELINE.json configs, SUSTAINED (each timed back to back for ~0.5 s) and at every N (each rank runs its own shard,
    the time is the max over ranks): Msamples/s whole-job and fraction of the per-GPU HBM roofline.  Plus the burst figure of the headline
    kernels (6 launches per interval, before the board reaches its power cap) for reference."""
    out = {"note": "sustained unless marked burst; Msamples/s are whole-job (all GPUs); frac = algorithmic bytes / time / (n_gpus x measured HBM peak)"}

    def entry(res):
        ms = _max_over_ranks(torch, dist, dev, res["ms"], distributed)
        val = n_gpus * res["samples_per_step"] / ms * 1e-3
        return {"workload": res["workload"], "steps": res.get("steps"), "ms_per_step": round(ms, 4), "value": round(val, 1), "unit": UNIT,
                "frac": round(res["bytes_per_sample"] * res["samples_per_step"] / (ms * 1e-3) * 1e-9 / peak, 4), "bytes_per_sample": res["bytes_per_sample"]}

    torch.cuda.synchronize()
    try:
        if n_gpus == 1:
            time.sleep(1.0)  # let the board leave the power-capped state of the main loop
            n = x.numel()
            y = mod(x)
            ta, ts = _burst(torch, lambda: mod(x)), _burst(torch, lambda: mod.inverse(y))
            out["n_band16_burst"] = {"analysis_ms": round(ta, 4), "synthesis_ms": round(ts, 4), "round_trip": round(n / (ta + ts) * 1e-3, 1),
                                     "frac": round(16 * n / ((ta + ts) * 1e-3) * 1e-9 / peak, 4)}
            del y
            out["single_stream_latency"] = bench_single_stream_latency(torch, pq, dev)
            # configs[0]: one clip of flute.wav's padded length (303 104 samples, batch 1), forward + inverse: launch-bound on a GPU
            x1 = (0.5 * torch.randn(1, 1, 303104, device=dev)).clamp_(-1, 1)
            t1, _ = _sustained(torch, lambda: mod.inverse(mod(x1)), 0.2, min_steps=50)
            out["config1"] = {"workload": "configs[0]: one 303 104-sample clip (flute.wav padded), n_band 16, forward + inverse, synthetic samples",
                              "ms_per_step": round(t1, 4), "value": round(303104 / t1 * 1e-3, 1), "unit": UNIT}
        out["config3"] = entry(bench_config3(torch, pq, dev, 0.5))
        r4 = bench_config4(torch, pq, dev, 2.0)
        per = {}
        for m, (ta, ts) in r4["per_band_ms"].items():
            ta = _max_over_ranks(torch, dist, dev, ta, distributed)
            ts = _max_over_ranks(torch, dist, dev, ts, distributed)
            per[f"n_band{m}"] = {"analysis_ms": round(ta, 4), "synthesis_ms": round(ts, 4), "value": round(n_gpus * r4["samples_per_step"] / (ta + ts) * 1e-3, 1),
                                 "unit": UNIT, "frac": round(16 * r4["samples_per_step"] / ((ta + ts) * 1e-3) * 1e-9 / peak, 4)}
        out["config4"] = {"workload": r4["workload"], "per_band": per}
        out["config5"] = entry(bench_config5(torch, pq, dev, 0.5))
    except Exception as exc:  # never let the informational part break the contract line
        out["error"] = repr(exc)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=("b200", "reference"), default="b200")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the sustained runs of configs 3 / 4 / 5 that are appended to the line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the sub-bands and reconstruction of the last step (rank 0, a fixed sample of rows) to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus > 1 and world == 1:
        # convenience: re-launch ourselves under torchrun (a launcher may also start torchrun itself)
        import subprocess

        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
               "--master-port", os.environ.get("MASTER_PORT", "29533"), os.path.abspath(__file__), "--gpus", str(args.gpus), "--steps",
               str(args.steps), "--warmup", str(args.warmup)] + (["--no-cpu-baseline"] if args.no_cpu_baseline else []) + (
                   ["--no-other-configs"] if args.no_other_configs else []) + (
                   ["--dump-outputs", os.path.abspath(args.dump_outputs)] if args.dump_outputs else [])
        return subprocess.call(cmd)
    return run_gpu(args)


if __name__ == "__main__":
    sys.exit(main())
