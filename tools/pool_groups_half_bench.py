"""Grouped stream-pool steps with bf16 / fp16 blocks (StreamPool(..., dtype).step_groups) against staging them on a float32 pool, against one
half-pool step per group and against the fp32 grouped step, in one process on one GPU (CUDA events, warm-up, arms alternated, medians
over rounds, with the range over the rounds).

Per n_band (16 / 8 / 32) and dtype, the workloads of tools/pool_groups_pcm_bench.py:
* A: four block lengths, every group just below the 96 tiles the streaming Hankel-4 kernels take alone;
* B: 1024 sessions at each of 512 / 1024 / 2048 / 4096 samples;
* C: A plus 200 sessions of 480-sample blocks (10 ms at 48 kHz), a group the kernels never plan: the grouped half call runs A natively and
  marks the 480-sample group for staging.
The arms, each one step_groups worth of work on every listed stream of the workload, with CUDA ids (a fixed random permutation):
    native     step_groups on the half pool (forward_groups, then inverse_groups of the rounded sub-bands)
    staged     on a float32 pool: widen, forward_groups, round, widen, inverse_groups, round -- what a half pool did before it had native
               grouped calls, and what the op does when the library refuses the call
    per_group  one half-pool step per group
    fp32       step_groups on a float32 pool, blocks widened once outside the timing: the yardstick
Prints the card and its power limit with the numbers."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import pqmf_b200 as pq
from pool_groups_pcm_bench import ROUNDS, INNER, alternate, card, streams_per_tile


def workloads(mod, m):
    """name -> [(sessions, T)]"""
    if m == 16:
        a = [(600, 512), (400, 1024), (250, 2048), (90, 4096)]
    else:
        lengths = (512, 1024, 2048, 4096) if m == 8 else (1024, 2048, 3072, 4096)
        a = [(95 * streams_per_tile(mod, T), T) for T in lengths]
    return {"A": a, "B": [(1024, T) for T in (512, 1024, 2048, 4096)], "C": a + [(200, 480)]}


def main():
    assert torch.cuda.is_available(), "pool_groups_half_bench needs a CUDA device"
    print(f"# {card()}")
    print(f"# ms per call, median [min, max] of {ROUNDS} alternating rounds x {INNER} calls")
    with torch.no_grad():
        for m in (16, 8, 32):
            mod = pq.CachedPQMF(100, m).cuda()
            for dtype in (torch.bfloat16, torch.float16):
                for name, shapes in workloads(mod, m).items():
                    P = sum(n for n, _ in shapes)
                    pool, fpool = pq.StreamPool(mod, P, dtype=dtype), pq.StreamPool(mod, P)
                    gen = torch.Generator(device="cuda").manual_seed(m)
                    perm = torch.randperm(P, device="cuda", generator=gen).to(torch.int32)
                    groups, r0 = [], 0
                    for n, T in shapes:
                        x = (0.5 * torch.randn(n, 1, T, device="cuda", generator=gen)).clamp_(-1, 1).to(dtype)
                        groups.append((x, perm[r0 : r0 + n].contiguous()))
                        r0 += n
                    fp = [(x.float(), i) for x, i in groups]

                    def staged():
                        ys = [y.to(dtype) for y in fpool.forward_groups([(x.float(), i) for x, i in groups])]
                        outs = [o.to(dtype) for o in fpool.inverse_groups([(y.float(), i) for y, (_, i) in zip(ys, groups)])]
                        return list(zip(outs, ys))

                    l0 = pq.launch_count()
                    pool.step_groups(groups)
                    native_launches = pq.launch_count() - l0
                    r = alternate({
                        "native": lambda: pool.step_groups(groups),
                        "staged": staged,
                        "per_group": lambda: [pool.step(x, i) for x, i in groups],
                        "fp32": lambda: fpool.step_groups(fp),
                    })
                    nat = r["native"][0]
                    arms = ", ".join(f"{k} {v[0]:.4f} [{v[1]:.4f}, {v[2]:.4f}] ms" for k, v in r.items())
                    print(f"n_band {m:2d} {str(dtype).split('.')[1]:8s} {name}: groups {shapes}: {arms}; native launches {native_launches}; "
                          f"staged / native {r['staged'][0] / nat:.2f}x, per_group / native {r['per_group'][0] / nat:.2f}x, "
                          f"fp32 / native {r['fp32'][0] / nat:.2f}x")


if __name__ == "__main__":
    main()
