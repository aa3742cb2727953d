"""Grouped stream-pool steps with 16-bit PCM blocks (StreamPool.step_groups_pcm16) against staging them, against one step_pcm16 per group
and against the fp32 grouped step, in one process on one GPU (CUDA events, warm-up, arms alternated, medians over rounds, with the range
over the rounds).

Per n_band (16 / 8 / 32), the workloads of tools/pool_groups_bench.py:
* A: four block lengths, every group just below the 96 tiles the streaming Hankel-4 kernels take alone (mono blocks);
* B: 1024 sessions at each of 512 / 1024 / 2048 / 4096 samples (mono blocks);
* B2: B with stereo blocks and downmix=True (one stream per clip);
* C: A plus 200 sessions of 480-sample blocks (10 ms at 48 kHz), a group the kernels never plan: the grouped PCM call runs A natively and
  marks the 480-sample group for staging.
The arms, each stepping every listed stream of the workload with CUDA ids (a fixed random permutation of the pool):
    native     step_groups_pcm16
    staged     widen each group (int16 -> float32 / 32768, the down-mix in channel order), step_groups, quantise each group -- what a caller
               without the grouped PCM call writes, and what the op does when the library refuses the call
    per_group  one step_pcm16 per group
    fp32       step_groups on float32 blocks (widened once, outside the timing): the yardstick
Prints the card and its power limit with the numbers."""
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
    """name -> ([(clips, T)], channels, downmix)"""
    if m == 16:
        a = [(600, 512), (400, 1024), (250, 2048), (90, 4096)]
    else:
        lengths = (512, 1024, 2048, 4096) if m == 8 else (1024, 2048, 3072, 4096)
        a = [(95 * streams_per_tile(mod, T), T) for T in lengths]
    b = [(1024, T) for T in (512, 1024, 2048, 4096)]
    return {"A": (a, 1, False), "B": (b, 1, False), "B2": (b, 2, True), "C": (a + [(200, 480)], 1, False)}


def widen(pcm, downmix):
    f = pcm.float().mul_(1.0 / 32768.0)
    if not downmix:
        return f.permute(0, 2, 1).reshape(-1, 1, pcm.shape[1])
    acc = f[..., 0].clone()
    for c in range(1, f.shape[-1]):
        acc.add_(f[..., c])
    return acc.div_(torch.full((), float(f.shape[-1]), device=acc.device)).unsqueeze(1)


def quantise(v, clips):
    return torch.clamp(torch.round(v * 32768.0), -32768.0, 32767.0).to(torch.int16).view(clips, -1, v.shape[-1]).permute(0, 2, 1).contiguous()


def main():
    assert torch.cuda.is_available(), "pool_groups_pcm_bench needs a CUDA device"
    print(f"# {card()}")
    print(f"# ms per call, median [min, max] of {ROUNDS} alternating rounds x {INNER} calls")
    with torch.no_grad():
        for m in (16, 8, 32):
            mod = pq.CachedPQMF(100, m).cuda()
            for name, (shapes, C, downmix) in workloads(mod, m).items():
                Cr = 1 if downmix else C
                P = sum(n * Cr for n, _ in shapes)
                pool = pq.StreamPool(mod, P)
                gen = torch.Generator(device="cuda").manual_seed(m)
                perm = torch.randperm(P, device="cuda", generator=gen).to(torch.int32)
                groups, r0 = [], 0
                for n, T in shapes:
                    pcm = (8000.0 * torch.randn(n, T, C, device="cuda", generator=gen)).round().clamp(-32768, 32767).to(torch.int16)
                    groups.append((pcm, perm[r0 : r0 + n * Cr].contiguous()))
                    r0 += n * Cr
                fp = [(widen(p, downmix), i) for p, i in groups]

                def staged():
                    res = pool.step_groups([(widen(p, downmix), i) for p, i in groups])
                    return [(quantise(o, p.shape[0]), y) for (o, y), (p, _) in zip(res, groups)]

                l0 = pq.launch_count()
                pool.step_groups_pcm16(groups, downmix=downmix)
                native_launches = pq.launch_count() - l0
                r = alternate({
                    "native": lambda: pool.step_groups_pcm16(groups, downmix=downmix),
                    "staged": staged,
                    "per_group": lambda: [pool.step_pcm16(p, i, downmix=downmix) for p, i in groups],
                    "fp32": lambda: pool.step_groups(fp),
                })
                nat = r["native"][0]
                arms = ", ".join(f"{k} {v[0]:.4f} [{v[1]:.4f}, {v[2]:.4f}] ms" for k, v in r.items())
                print(f"n_band {m:2d} {name}: groups {shapes} x {C} ch{' down-mixed' if downmix else ''}: {arms}; native launches "
                      f"{native_launches}; staged / native {r['staged'][0] / nat:.2f}x, per_group / native {r['per_group'][0] / nat:.2f}x, "
                      f"fp32 / native {r['fp32'][0] / nat:.2f}x")


if __name__ == "__main__":
    main()
