"""Device-side timing of the half-precision I/O (CUDA events per call, inputs larger than the 126 MB L2): fp32, native bf16 (the
half-precision Hankel-4 kernels) and staged bf16 (cast to fp32, fp32 kernel, cast back -- what a caller without native half I/O
runs), alternated in one process; medians over the rounds.  n_band 16 at 64 x 2^20, n_band 4 / 8 / 32 at bench.py's config-4 shape
(64 x 2 880 000).  Prints the card and its power limit with the numbers."""
import os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import statistics
import torch
import pqmf_b200 as pq

ROUNDS, INNER = 9, 8


def per_call_ms(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(INNER):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / INNER


def card():
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # pragma: no cover
        limit = f"unknown ({e})"
    return f"{torch.cuda.get_device_name()}, power limit {limit}"


def main():
    assert torch.cuda.is_available(), "half_bench needs a CUDA device"
    print(f"# {card()}")
    print(f"# ms per call, median of {ROUNDS} alternating rounds x {INNER} calls; native / staged relative to fp32 and to each other")
    bf = torch.bfloat16
    for m, rows, t in [(16, 64, 1 << 20), (4, 64, 2_880_000), (8, 64, 2_880_000), (32, 64, 2_880_000)]:
        mod = pq.PQMF(100, m).cuda()
        gen = torch.Generator(device="cuda").manual_seed(m)
        x32 = (0.5 * torch.randn(rows, 1, t, device="cuda", generator=gen)).clamp_(-1, 1)
        xb = x32.to(bf)
        y32, yb = mod(x32), mod(xb)
        assert torch.equal(yb.view(torch.int16), mod(xb.float()).to(bf).view(torch.int16))
        variants = {
            "analysis": {"fp32": lambda: mod(x32), "bf16 native": lambda: mod(xb), "bf16 staged": lambda: mod(xb.float()).to(bf)},
            "synthesis": {"fp32": lambda: mod.inverse(y32), "bf16 native": lambda: mod.inverse(yb),
                          "bf16 staged": lambda: mod.inverse(yb.float()).to(bf)},
        }
        for direction, fns in variants.items():
            times = {k: [] for k in fns}
            for fn in fns.values():  # warm-up
                fn()
            torch.cuda.synchronize()
            for _ in range(ROUNDS):
                for k, fn in fns.items():
                    times[k].append(per_call_ms(fn))
            med = {k: statistics.median(v) for k, v in times.items()}
            spread = {k: (max(v) - min(v)) / med[k] for k, v in times.items()}
            print(f"n_band {m:2d} {rows} x {t} {direction:9s}  fp32 {med['fp32']:.4f}  bf16 native {med['bf16 native']:.4f}  "
                  f"bf16 staged {med['bf16 staged']:.4f}  native/fp32 {med['bf16 native'] / med['fp32']:.3f}  "
                  f"native/staged {med['bf16 native'] / med['bf16 staged']:.3f}  (spread {max(spread.values()):.1%})")
        del x32, xb, y32, yb, mod
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
