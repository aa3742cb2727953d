"""Half-precision stream-pool steps (StreamPool(mod, P, dtype=torch.bfloat16 / torch.float16).step) against staging them and against the
float32 pool step, in one process on one GPU (CUDA events, warm-up, arms alternated, medians over rounds, with the range over the rounds).

One pool step of 4096 sessions x 2048 samples at n_band 8 / 16 / 32, with ids = arange(4096) and with a random half of a pool of 8192
(CUDA ids, fixed per workload).  The arms:
    native  step on the half pool: the streaming Hankel-4 POOL kernels with half loads and stores (3 launches)
    staged  on a float32 pool: widen, forward, round, widen, inverse, round -- what a caller without half pools writes, and what the op
            does where the library has no native kernel
    fp32    step on the float32 pool with float32 blocks (widened once, outside the timing): the yardstick
Native half moves 12 B/sample through HBM (2 in, 4 + 2 sub-bands, 2 out, plus the state) against 20 for fp32 and more for staging.
Prints the card and its power limit with the numbers."""
import os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import statistics
import torch
import pqmf_b200 as pq

ROUNDS, INNER = 11, 20
B, T = 4096, 2048


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
    for fn in arms.values():  # warm-up: module loads, shared-memory opt-ins
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for _ in range(ROUNDS):
        for k, fn in arms.items():
            times[k].append(per_call_ms(fn))
    return {k: (statistics.median(v), min(v), max(v)) for k, v in times.items()}


def main():
    assert torch.cuda.is_available(), "pool_half_bench needs a CUDA device"
    print(f"# {card()}")
    print(f"# one pool step of {B} sessions x {T} samples; ms per call, median [min, max] of {ROUNDS} alternating rounds x {INNER} calls")
    with torch.no_grad():
        for m in (8, 16, 32):
            mod = pq.CachedPQMF(100, m).cuda()
            for ids_name, P in (("arange", B), ("random half", 2 * B)):
                gen = torch.Generator(device="cuda").manual_seed(m)
                ids = (torch.arange(B, device="cuda") if P == B else torch.randperm(P, device="cuda", generator=gen)[:B]).to(torch.int32)
                for dtype in (torch.bfloat16, torch.float16):
                    half, full = pq.StreamPool(mod, P, dtype=dtype), pq.StreamPool(mod, P)
                    x = (0.5 * torch.randn(B, 1, T, device="cuda", generator=gen)).clamp_(-1, 1).to(dtype)
                    xf = x.float()

                    def staged():
                        y = full.forward(x.float(), ids).to(dtype)
                        return full.inverse(y.float(), ids).to(dtype), y

                    l0 = pq.launch_count()
                    half.step(x, ids)
                    launches = pq.launch_count() - l0
                    r = alternate({"native": lambda: half.step(x, ids), "staged": staged, "fp32": lambda: full.step(xf, ids)})
                    nat = r["native"][0]
                    arms = ", ".join(f"{k} {v[0]:.4f} [{v[1]:.4f}, {v[2]:.4f}] ms" for k, v in r.items())
                    print(f"n_band {m:2d} {str(dtype)[6:]:8s} ids {ids_name:11s}: {arms}; native launches {launches}; "
                          f"staged / native {r['staged'][0] / nat:.2f}x, fp32 / native {r['fp32'][0] / nat:.2f}x")


if __name__ == "__main__":
    main()
