"""Stream pools against lockstep streaming, in one process on one GPU (CUDA events, warm-up, arms alternated, medians over rounds).

* n_band 16 / 8 / 32, 4096 streams x 2048-sample blocks: CachedPQMF.process_stream (lockstep), StreamPool.step with ids = arange(4096),
  and StreamPool.step on a random 2048 of the 4096 streams (a new draw every call); reported per block step and per stream-block.
  The arms run back to back on the same buffers (inputs, outputs and state together are about the size of the 126 MB L2).
* single-stream latency, 512- and 4096-sample blocks: a graph-replayed StreamPool.step against StreamGraph.
Prints the card and its power limit with the numbers."""
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


def main():
    assert torch.cuda.is_available(), "pool_bench needs a CUDA device"
    print(f"# {card()}")
    print(f"# ms per call, median of {ROUNDS} alternating rounds x {INNER} calls")
    S, T = 4096, 2048
    with torch.no_grad():
        for m in (16, 8, 32):
            mod = pq.CachedPQMF(100, m).cuda()
            pool = pq.StreamPool(mod, S)
            gen = torch.Generator(device="cuda").manual_seed(m)
            x = (0.5 * torch.randn(S, 1, T, device="cuda", generator=gen)).clamp_(-1, 1)
            half = x[: S // 2].contiguous()
            ids = torch.arange(S, device="cuda", dtype=torch.int32)
            draws = [torch.randperm(S, device="cuda", generator=gen)[: S // 2].to(torch.int32) for _ in range(16)]
            k = [0]

            def subset():
                k[0] += 1
                return pool.step(half, draws[k[0] % len(draws)])

            r = alternate({"lockstep": lambda: mod.process_stream(x), "pool": lambda: pool.step(x, ids), "pool_half": subset})
            print(f"n_band {m:2d}, {S} x {T}: lockstep {r['lockstep']:.4f} ms, pool arange {r['pool']:.4f} ms "
                  f"({100 * (r['pool'] / r['lockstep'] - 1):+.1f} %), pool random {S // 2} {r['pool_half']:.4f} ms | per stream-block: "
                  f"lockstep {1e6 * r['lockstep'] / S:.2f} ns, pool {1e6 * r['pool'] / S:.2f} ns, pool random half {1e6 * r['pool_half'] / (S // 2):.2f} ns")
        for block in (512, 4096):
            mod = pq.CachedPQMF(100, 16).cuda()
            sg = pq.StreamGraph(pq.CachedPQMF(100, 16).cuda(), 1, block)
            pool = pq.StreamPool(mod, 64)
            sx = torch.zeros(1, 1, block, device="cuda")
            sid = torch.tensor([5], device="cuda", dtype=torch.int32)
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                pool.step(sx, sid)
            torch.cuda.current_stream().wait_stream(side)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                pool.step(sx, sid)
            r = alternate({"stream_graph": lambda: sg.step(), "pool_graph": g.replay})
            print(f"1 stream x {block}: StreamGraph {1e3 * r['stream_graph']:.1f} us, graph-replayed pool step {1e3 * r['pool_graph']:.1f} us per block "
                  f"(back-to-back replays)")


if __name__ == "__main__":
    main()
