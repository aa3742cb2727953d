"""int16 PCM blocks in the streaming calls against staging them and against float32 blocks, in one process on one GPU (CUDA events,
warm-up, arms alternated, medians over rounds).

* n_band 16 / 8 / 32, 4096 mono streams x 2048-sample blocks, lockstep (CachedPQMF.process_stream_pcm16) and in a pool (StreamPool.step_pcm16,
  ids = arange(4096)), per block step:
    native  the streaming Hankel-4 kernels with PCM loads and stores (the PCM call itself)
    staged  widen (int16 -> float32 / 32768), the float32 step, quantise -- what a caller without the PCM entries does
    fp32    the float32 step on float32 blocks
* end to end, per arm: a pinned host block -> H2D copy -> step -> D2H copy of the output block, float32 against PCM (plain async copies on
  the current stream).
Each arm has its own module / pool, so the arms do not share state.  Prints the card and its power limit with the numbers."""
import os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import statistics
import torch
import pqmf_b200 as pq

ROUNDS, INNER = 11, 20


def per_call_ms(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(INNER):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / INNER


def card():
    # by UUID: torch's device index is not nvidia-smi's index under CUDA_VISIBLE_DEVICES
    try:
        uuid = f"GPU-{torch.cuda.get_device_properties(torch.cuda.current_device()).uuid}"
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", uuid],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # pragma: no cover
        q = f"{torch.cuda.get_device_name()}, power limit unknown ({e})"
    return q


def alternate(arms):
    for fn in arms.values():  # warm-up: module loads, shared-memory opt-ins, state allocation
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for _ in range(ROUNDS):
        for k, fn in arms.items():
            times[k].append(per_call_ms(fn))
    return {k: statistics.median(v) for k, v in times.items()}


def widen(pcm):  # mono [S, T, 1] -> [S, 1, T]
    return pcm.view(pcm.shape[0], 1, pcm.shape[1]).to(torch.float32).mul_(1.0 / 32768.0)


def quantise(out):  # [S, 1, T] -> [S, T, 1]
    return (out * 32768.0).round_().clamp_(-32768, 32767).to(torch.int16).view(out.shape[0], out.shape[2], 1)


def launches(fn):
    n0 = pq.launch_count()
    fn()
    return pq.launch_count() - n0


def main():
    assert torch.cuda.is_available(), "stream_pcm_bench needs a CUDA device"
    print(f"# {card()}")
    print(f"# ms per block step, median of {ROUNDS} alternating rounds x {INNER} calls; mono blocks")
    S, T = 4096, 2048
    with torch.no_grad():
        for m in (16, 8, 32):
            gen = torch.Generator(device="cuda").manual_seed(m)
            pcm = (8000.0 * torch.randn(S, T, 1, device="cuda", generator=gen)).round_().clamp_(-32768, 32767).to(torch.int16)
            x = widen(pcm)
            ids = torch.arange(S, device="cuda", dtype=torch.int32)
            mods = {k: pq.CachedPQMF(100, m).cuda() for k in ("native", "staged", "fp32")}
            pools = {k: pq.StreamPool(pq.CachedPQMF(100, m).cuda(), S) for k in ("native", "staged", "fp32")}
            arms = {
                "lockstep native": lambda: mods["native"].process_stream_pcm16(pcm),
                "lockstep staged": lambda: quantise(mods["staged"].process_stream(widen(pcm))[0]),
                "lockstep fp32": lambda: mods["fp32"].process_stream(x),
                "pool native": lambda: pools["native"].step_pcm16(pcm, ids),
                "pool staged": lambda: quantise(pools["staged"].step(widen(pcm), ids)[0]),
                "pool fp32": lambda: pools["fp32"].step(x, ids),
            }
            n_native = (launches(arms["lockstep native"]), launches(arms["pool native"]))
            n_fp32 = (launches(arms["lockstep fp32"]), launches(arms["pool fp32"]))
            r = alternate(arms)
            for kind in ("lockstep", "pool"):
                nat, stg, f32 = r[f"{kind} native"], r[f"{kind} staged"], r[f"{kind} fp32"]
                print(f"n_band {m:2d}, {S} x {T}, {kind:8s}: native PCM {nat:.4f} ms, staged PCM {stg:.4f} ms ({100 * (stg / nat - 1):+.1f} % vs native), "
                      f"fp32 {f32:.4f} ms (native PCM {100 * (nat / f32 - 1):+.1f} % vs fp32)")
            print(f"  library launches per step: native PCM lockstep {n_native[0]}, pool {n_native[1]}; fp32 lockstep {n_fp32[0]}, pool {n_fp32[1]}")
            # end to end: pinned host block in, pinned host block out
            h_pcm, h_x = pcm.cpu().pin_memory(), x.cpu().pin_memory()
            d_pcm, d_x = torch.empty_like(pcm), torch.empty_like(x)
            o_pcm = torch.empty(S, T, 1, dtype=torch.int16).pin_memory()
            o_x = torch.empty(S, 1, T).pin_memory()

            def e2e(kind, fmt):
                def run():
                    if fmt == "pcm":
                        d_pcm.copy_(h_pcm, non_blocking=True)
                        out = mods["native"].process_stream_pcm16(d_pcm)[0] if kind == "lockstep" else pools["native"].step_pcm16(d_pcm, ids)[0]
                        o_pcm.copy_(out, non_blocking=True)
                    else:
                        d_x.copy_(h_x, non_blocking=True)
                        out = mods["fp32"].process_stream(d_x)[0] if kind == "lockstep" else pools["fp32"].step(d_x, ids)[0]
                        o_x.copy_(out, non_blocking=True)
                return run

            r = alternate({f"{k} {f}": e2e(k, f) for k in ("lockstep", "pool") for f in ("fp32", "pcm")})
            for kind in ("lockstep", "pool"):
                f32, p16 = r[f"{kind} fp32"], r[f"{kind} pcm"]
                print(f"  end to end {kind:8s} (H2D, step, D2H): fp32 {f32:.4f} ms = {S * T / f32 / 1e6:.2f} Gsamples/s, "
                      f"PCM {p16:.4f} ms = {S * T / p16 / 1e6:.2f} Gsamples/s ({100 * (p16 / f32 - 1):+.1f} %)")


if __name__ == "__main__":
    main()
