"""Grouped stream-pool steps (StreamPool.step_groups) against one StreamPool.step per group, in one process on one GPU (CUDA events,
warm-up, arms alternated, medians over rounds, with the range over the rounds).

Per n_band (16 / 8 / 32), two workloads of four block lengths each:
* A: every group just below the 96 tiles the streaming Hankel-4 kernels take alone (n_band 16: the 600 / 400 / 250 / 90 sessions at
  512 / 1024 / 2048 / 4096 samples; n_band 8 / 32: 95 tiles' worth of streams per block length, from the plan's streams per tile), so
  one call per group runs the direct form and the grouped call runs them together on the tensor cores;
* B: 1024 sessions at each of 512 / 1024 / 2048 / 4096 samples, so every group the kernels can plan is native on its own.
Every call steps all the listed streams of one workload with CUDA ids (a fixed random permutation of the pool).  Prints the card and
its power limit with the numbers."""
import os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import statistics
import torch
import pqmf_b200 as pq

ROUNDS, INNER = 11, 20
FLAG_BLOCKERS = 2 | 4 | 8 | 16 | (1 << 23)


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


def streams_per_tile(mod, T):
    """Streams per MMA tile of a T-sample block on the streaming Hankel-4 kernels (the plan in pqmf_b200.cu), or None."""
    m, length = mod.hk.shape
    flags = mod._flags
    jlo, kt = 32 * ((flags >> 8) & 0xF), 32 * ((flags >> 12) & 0x1F)
    if m not in (8, 16, 32) or mod._tables.numel() == 0 or kt == 0 or flags & FLAG_BLOCKERS or T % 256 or T < length:
        return None
    hist = max(-(-(length - jlo) // 64) * 64, -(-(jlo + kt) // 64) * 64)
    pitch = (T // 64 + hist // 64 + 3) & ~3
    return 128 // pitch if pitch <= 128 else None


def workloads(mod, m):
    if m == 16:
        a = [(600, 512), (400, 1024), (250, 2048), (90, 4096)]
    else:
        lengths = (512, 1024, 2048, 4096) if m == 8 else (1024, 2048, 3072, 4096)
        a = [(95 * streams_per_tile(mod, T), T) for T in lengths]
    b = [(1024, T) for T in (512, 1024, 2048, 4096)]
    return {"A": a, "B": b}


def main():
    assert torch.cuda.is_available(), "pool_groups_bench needs a CUDA device"
    print(f"# {card()}")
    print(f"# ms per call, median [min, max] of {ROUNDS} alternating rounds x {INNER} calls")
    with torch.no_grad():
        for m in (16, 8, 32):
            mod = pq.CachedPQMF(100, m).cuda()
            for name, shapes in workloads(mod, m).items():
                P = sum(n for n, _ in shapes)
                pool = pq.StreamPool(mod, P)
                gen = torch.Generator(device="cuda").manual_seed(m)
                perm = torch.randperm(P, device="cuda", generator=gen).to(torch.int32)
                groups, r0 = [], 0
                for n, T in shapes:
                    groups.append(((0.5 * torch.randn(n, 1, T, device="cuda", generator=gen)).clamp_(-1, 1), perm[r0 : r0 + n].contiguous()))
                    r0 += n
                l0 = pq.launch_count()
                pool.step_groups(groups)
                grouped_launches = pq.launch_count() - l0
                r = alternate({"grouped": lambda: pool.step_groups(groups), "sequential": lambda: [pool.step(x, i) for x, i in groups]})
                tiles = [(-(-n // s) if s else None) for (n, T), s in zip(shapes, (streams_per_tile(mod, T) for _, T in shapes))]
                g, s = r["grouped"], r["sequential"]
                print(f"n_band {m:2d} {name}: groups {shapes} (tiles alone {tiles}): grouped {g[0]:.4f} [{g[1]:.4f}, {g[2]:.4f}] ms "
                      f"({grouped_launches} launches), sequential {s[0]:.4f} [{s[1]:.4f}, {s[2]:.4f}] ms ({3 * len(shapes)} launches): "
                      f"{s[0] / g[0]:.2f}x")


if __name__ == "__main__":
    main()
