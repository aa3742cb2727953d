"""int16 PCM blocks in the streaming calls: CachedPQMF.forward_stream_pcm16 / inverse_stream_pcm16 / process_stream_pcm16 and
StreamPool.step_pcm16 / forward_pcm16 / inverse_pcm16.

Every PCM call must give the bits of its float32 counterpart on the widened block (v / 32768 per channel; the down-mix summed in channel
order, then / C), followed by the quantisation clamp(rint(v * 32768), -32768, 32767), with the same state, slot, frame-counter, pool and
phase-word updates -- whether it runs the streaming Hankel-4 kernels with PCM loads and stores or is staged through the float32 op.  The
last test needs no GPU: it checks the C entries' argument validation."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import pqmf_oracle as O

ERR_ARG, ERR_UNSUPPORTED = -1, -2


@pytest.fixture(scope="module")
def pq():
    import pqmf_b200

    return pqmf_b200


def widen(pcm, downmix):
    """[S, T, C] int16 -> [S, C', T] float32, the kernels' arithmetic (a tensor divisor: torch divides by a host scalar via its reciprocal)."""
    f = pcm.to(torch.float32) * (1.0 / 32768.0)
    if not downmix:
        return f.permute(0, 2, 1).contiguous()
    acc = f[..., 0].clone()
    for c in range(1, f.shape[-1]):
        acc += f[..., c]
    return (acc / torch.tensor(float(f.shape[-1]), device=acc.device)).unsqueeze(1)


def quantise(v):
    """[S, C, T] float32 -> [S, T, C] int16."""
    return (v * 32768.0).round().clamp(-32768, 32767).to(torch.int16).permute(0, 2, 1).contiguous()


def pcm_blocks(shape, seed, device="cuda"):
    g = torch.Generator(device=device).manual_seed(seed)
    return (8000.0 * torch.randn(shape, device=device, generator=g)).round().clamp(-32768, 32767).to(torch.int16)


def same_state(a, b):
    return (torch.equal(a._x_state, b._x_state) and torch.equal(a._s_state, b._s_state) and a._x_slot == b._x_slot and a._s_slot == b._s_slot
            and a._frames_in == b._frames_in and a._frames_out == b._frames_out)


# (n_band, blocks, channels, downmix): 300 rows of 2048 samples = at least 100 tiles of the streaming Hankel-4 kernels at n_band 8 / 16 / 32
LOCKSTEP = [(m, s, c, d) for m in (8, 16, 32) for (s, c, d) in ((300, 1, False), (150, 2, False), (300, 2, True))]


@pytest.mark.gpu
@pytest.mark.parametrize("m,S,C,downmix", LOCKSTEP)
def test_lockstep_equals_fp32_twin(pq, m, S, C, downmix):
    """Native blocks interleaved with a 3-frame PCM block (staged) and a float32 block on the same module, so the native kernels run at
    both frame parities; split calls and one-op steps alternate.  Outputs, both state halves, slots and frame counters equal the twin's."""
    mod, twin = pq.CachedPQMF(100, m).cuda(), pq.CachedPQMF(100, m).cuda()
    T = 2048
    plan = ["step", "split", "3frames", "step", "fp32", "split", "step"]
    for k, kind in enumerate(plan):
        if kind == "fp32":
            x = (0.5 * torch.randn(S * (1 if downmix else C), 1, T, device="cuda")).clamp_(-1, 1)
            a, b = mod.process_stream(x), twin.process_stream(x)
            assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and same_state(mod, twin), k
            continue
        t = 3 * m if kind == "3frames" else T
        pcm = pcm_blocks((S, t, C), 100 * m + k)
        xw = widen(pcm, downmix)
        if kind == "split":
            y = mod.forward_stream_pcm16(pcm, downmix)
            out = mod.inverse_stream_pcm16(y)
        else:
            out, y = mod.process_stream_pcm16(pcm, downmix)
        out_r, y_r = twin.process_stream(xw)
        assert y.dtype == torch.float32 and out.dtype == torch.int16
        assert torch.equal(y, y_r.view(y.shape)), (k, kind)
        assert torch.equal(out, quantise(out_r)), (k, kind)
        assert same_state(mod, twin), (k, kind)


@pytest.mark.gpu
@pytest.mark.parametrize("route", ("fold", "direct", "misaligned"))
def test_staged_routes_equal_fp32_twin(pq, route):
    """Calls the streaming Hankel-4 kernels do not serve: few n_band-16 streams (fold kernels), n_band 4 (direct form), a misaligned view."""
    m, S, C = {"fold": (16, 7, 2), "direct": (4, 5, 2), "misaligned": (16, 300, 1)}[route]
    mod, twin = pq.CachedPQMF(100, m).cuda(), pq.CachedPQMF(100, m).cuda()
    for k in range(3):
        pcm = pcm_blocks((S, 2048, C), 7 * k + m)
        if route == "misaligned":  # a contiguous view 2 bytes past an aligned address
            buf = torch.empty(pcm.numel() + 16, dtype=torch.int16, device="cuda")
            pcm = buf[1 : 1 + pcm.numel()].view(pcm.shape).copy_(pcm)
            assert pcm.data_ptr() % 32 != 0 and pcm.is_contiguous()
        out, y = mod.process_stream_pcm16(pcm)
        out_r, y_r = twin.process_stream(widen(pcm, False))
        assert torch.equal(y, y_r.view(y.shape)) and torch.equal(out, quantise(out_r)) and same_state(mod, twin), (route, k)


def _cabi(pq):
    c = pq._lib.cabi
    vp, i, lg, u = ctypes.c_void_p, ctypes.c_int, ctypes.c_long, ctypes.c_uint
    c.pqmf_analysis_stream_pcm16.argtypes = [vp] * 6 + [i, lg, i, i, i, i, i, u, vp]
    c.pqmf_synthesis_stream_pcm16.argtypes = [vp] * 6 + [i, i, lg, i, i, i, u, vp]
    c.pqmf_stream_step_pcm16.argtypes = [vp] * 9 + [i, lg, i, i, i, i, i, i, u, vp]
    c.pqmf_stream_pool_analysis_pcm16.argtypes = [vp] * 6 + [i, vp, i, lg, i, i, i, i, u, vp]
    c.pqmf_stream_pool_synthesis_pcm16.argtypes = [vp] * 6 + [i, vp, i, i, lg, i, i, u, vp]
    c.pqmf_stream_pool_step_pcm16.argtypes = [vp] * 9 + [i, vp, i, lg, i, i, i, i, u, vp]
    for f in ("analysis_stream", "synthesis_stream", "stream_step", "stream_pool_analysis", "stream_pool_synthesis", "stream_pool_step"):
        getattr(c, f"pqmf_{f}_pcm16").restype = ctypes.c_int
    return c


@pytest.mark.gpu
@pytest.mark.parametrize("m", (8, 16, 32))
def test_cabi_native_or_refused_before_launching(pq, m):
    """The C entries return 0 on the native shapes and PQMF_ERR_UNSUPPORTED, with no launch and no state written, on the staged ones:
    the PCM instantiations of every band count run where the twin tests above expect them to."""
    c = _cabi(pq)
    mod = pq.CachedPQMF(100, m).cuda()
    hk, tab, M, L, fl = mod.hk, mod._tables, m, mod.hk.shape[1], mod._flags
    st = torch.cuda.current_stream().cuda_stream

    def run(S, T, C, downmix, offset=0):
        rows = S * (1 if downmix else C)
        buf = pcm_blocks((S * T * C + 16,), S + T)
        pcm = buf[offset:]
        y = torch.zeros(rows, M, T // M, device="cuda")
        obuf = torch.zeros(S * T * (1 if downmix else C) + 16, dtype=torch.int16, device="cuda")
        out = obuf[offset : offset + S * T * (1 if downmix else C)].view(S, T, 1 if downmix else C)
        xs = [torch.zeros(rows, L, device="cuda") for _ in range(2)]
        ss = [torch.zeros(rows, L, device="cuda") for _ in range(2)]
        xs[0].normal_()
        ss[0].normal_()
        ids = torch.arange(rows, dtype=torch.int32, device="cuda")
        P = max(rows, 1)
        xpool, spool = torch.randn(2, P, L, device="cuda"), torch.randn(2, P, L, device="cuda")
        xph, sph = torch.zeros(P, dtype=torch.int32, device="cuda"), torch.zeros(P, dtype=torch.int32, device="cuda")
        snap = [t.clone() for t in (xs[1], ss[1], y, out, xpool, spool, xph, sph)]
        d = 1 if downmix else 0
        rcs = {}
        n0 = pq.launch_count()
        rcs["analysis"] = (c.pqmf_analysis_stream_pcm16(pcm.data_ptr(), y.data_ptr(), hk.data_ptr(), tab.data_ptr(), xs[0].data_ptr(), xs[1].data_ptr(),
                                                         S, T, C, d, M, L, 0, fl, st), pq.launch_count() - n0)
        n0 = pq.launch_count()
        rcs["synthesis"] = (c.pqmf_synthesis_stream_pcm16(y.data_ptr(), out.data_ptr(), hk.data_ptr(), tab.data_ptr(), ss[0].data_ptr(), ss[1].data_ptr(),
                                                          S, 1 if downmix else C, T // M, M, L, 0, fl, st), pq.launch_count() - n0)
        n0 = pq.launch_count()
        rcs["step"] = (c.pqmf_stream_step_pcm16(pcm.data_ptr(), y.data_ptr(), out.data_ptr(), hk.data_ptr(), tab.data_ptr(), xs[0].data_ptr(),
                                                xs[1].data_ptr(), ss[0].data_ptr(), ss[1].data_ptr(), S, T, C, d, M, L, 0, 0, fl, st), pq.launch_count() - n0)
        n0 = pq.launch_count()
        rcs["pool_analysis"] = (c.pqmf_stream_pool_analysis_pcm16(pcm.data_ptr(), y.data_ptr(), hk.data_ptr(), tab.data_ptr(), xpool.data_ptr(),
                                                                  xph.data_ptr(), P, ids.data_ptr(), S, T, C, d, M, L, fl, st), pq.launch_count() - n0)
        n0 = pq.launch_count()
        rcs["pool_synthesis"] = (c.pqmf_stream_pool_synthesis_pcm16(y.data_ptr(), out.data_ptr(), hk.data_ptr(), tab.data_ptr(), spool.data_ptr(),
                                                                    sph.data_ptr(), P, ids.data_ptr(), S, 1 if downmix else C, T // M, M, L, fl, st),
                                 pq.launch_count() - n0)
        n0 = pq.launch_count()
        rcs["pool_step"] = (c.pqmf_stream_pool_step_pcm16(pcm.data_ptr(), y.data_ptr(), out.data_ptr(), hk.data_ptr(), tab.data_ptr(), xpool.data_ptr(),
                                                          xph.data_ptr(), spool.data_ptr(), sph.data_ptr(), P, ids.data_ptr(), S, T, C, d, M, L, fl, st),
                            pq.launch_count() - n0)
        torch.cuda.synchronize()
        untouched = all(torch.equal(a, b) for a, b in zip(snap, (xs[1], ss[1], y, out, xpool, spool, xph, sph)))
        return rcs, untouched

    native_launches = {"analysis": 1, "synthesis": 1, "step": 2, "pool_analysis": 2, "pool_synthesis": 2, "pool_step": 3}
    for shape in ((300, 2048, 1, False), (300, 2048, 2, True)):
        rcs, _ = run(*shape)
        assert rcs == {k: (0, v) for k, v in native_launches.items()}, (shape, rcs)
    # stereo rows: native analysis, interleaved output staged
    rcs, _ = run(150, 2048, 2, False)
    assert rcs["analysis"] == (0, 1) and rcs["pool_analysis"] == (0, 2), rcs
    assert all(rcs[k] == (ERR_UNSUPPORTED, 0) for k in ("synthesis", "step", "pool_synthesis", "pool_step")), rcs
    # staged shapes: nothing launched, nothing written
    for shape, offset in (((300, 3 * M, 1, False), 0), ((7, 2048, 1, False), 0), ((300, 2048, 1, False), 1)):
        rcs, untouched = run(*shape, offset=offset)
        assert all(v == (ERR_UNSUPPORTED, 0) for v in rcs.values()) and untouched, (shape, offset, rcs)
    if m != 16:
        return
    # n_band 4: the direct form
    mod4 = pq.CachedPQMF(100, 4).cuda()
    L4 = mod4.hk.shape[1]
    pcm = pcm_blocks((300, 2048, 1), 3)
    y = torch.zeros(300, 4, 512, device="cuda")
    xs = [torch.zeros(300, L4, device="cuda") for _ in range(2)]
    n0 = pq.launch_count()
    assert c.pqmf_analysis_stream_pcm16(pcm.data_ptr(), y.data_ptr(), mod4.hk.data_ptr(), mod4._tables.data_ptr(), xs[0].data_ptr(), xs[1].data_ptr(),
                                        300, 2048, 1, 0, 4, L4, 0, mod4._flags, st) == ERR_UNSUPPORTED
    assert pq.launch_count() == n0


@pytest.mark.gpu
def test_full_scale_and_saturation(pq):
    """Inputs at -32768 / 32767, and sub-bands scaled so that the reconstruction clips: equal to the torch quantisation of the fp32 result."""
    m, S = 16, 300
    mod, twin = pq.CachedPQMF(100, m).cuda(), pq.CachedPQMF(100, m).cuda()
    g = torch.Generator(device="cuda").manual_seed(5)
    for k in range(3):
        pcm = torch.where(torch.rand(S, 2048, 1, device="cuda", generator=g) < 0.5, -32768, 32767).to(torch.int16)
        pcm[:, :: 7 + k] = 0
        out, y = mod.process_stream_pcm16(pcm)
        out_r, y_r = twin.process_stream(widen(pcm, False))
        assert torch.equal(y, y_r) and torch.equal(out, quantise(out_r)) and same_state(mod, twin)
    clipped = 0
    for k in range(3):
        s = 4.0 * torch.randn(S, m, 128, device="cuda", generator=g)
        out = mod.inverse_stream_pcm16(s)
        want = quantise(twin.inverse_stream(s))
        assert torch.equal(out, want) and same_state(mod, twin), k
        clipped += int(((out == 32767) | (out == -32768)).sum())
    assert clipped > 1000


def _widened_rows(pcm, downmix):
    x = widen(pcm, downmix)
    return x.reshape(-1, 1, x.shape[-1])


@pytest.mark.gpu
def test_pool_schedule_equals_fp32_twin(pq):
    """A seeded 12-step schedule over a pool of 4096: random subsets and orders, stereo ids, down-mix steps, a reset, native and staged
    shapes.  After every step the pool buffers, both phase-word arrays and the outputs equal a twin pool stepped with pool.step on the widened
    blocks, and streams not stepped are unchanged."""
    P, m = 4096, 16
    mod = pq.CachedPQMF(100, m).cuda()
    pool, twin = pq.StreamPool(mod, P), pq.StreamPool(mod, P)
    rng = np.random.default_rng(77)
    schedule = [(4096, 2048, 1, False), (150, 2048, 2, False), (300, 2048, 2, True), (2000, 48, 1, False), ("reset", 0, 0, False),
                (1500, 2048, 2, False), (40, 2048, 1, False), (1000, 2048, 3, True), (700, 2048, 3, False), (4096, 48, 1, False),
                (2048, 2048, 2, False), (7, 2048, 2, True)]
    for step, (S, T, C, downmix) in enumerate(schedule):
        if S == "reset":
            gone = rng.choice(P, 700, replace=False).tolist()
            pool.reset(gone)
            twin.reset(gone)
            continue
        rows = S * (1 if downmix else C)
        ids = torch.from_numpy(rng.choice(P, rows, replace=False).astype(np.int32)).cuda()
        pcm = pcm_blocks((S, T, C), 1000 + step)
        before = [t.clone() for t in (pool.xpool, pool.spool, pool.xphase, pool.sphase)]
        out, y = pool.step_pcm16(pcm, ids if step % 2 else ids.tolist(), downmix)
        out_r, y_r = twin.step(_widened_rows(pcm, downmix), ids)
        Cr = 1 if downmix else C
        assert torch.equal(y, y_r.view(S, Cr * m, T // m)), step
        assert torch.equal(out, quantise(out_r.view(S, Cr, T))), step
        for u, v in zip((pool.xpool, pool.spool, pool.xphase, pool.sphase), (twin.xpool, twin.spool, twin.xphase, twin.sphase)):
            assert torch.equal(u, v), step
        rest = torch.ones(P, dtype=torch.bool, device="cuda")
        rest[ids.long()] = False
        assert torch.equal(pool.xpool[:, rest], before[0][:, rest]) and torch.equal(pool.spool[:, rest], before[1][:, rest]), step
        assert torch.equal(pool.xphase[rest], before[2][rest]) and torch.equal(pool.sphase[rest], before[3][rest]), step


@pytest.mark.gpu
@pytest.mark.parametrize("m,S,C,downmix", ((16, 300, 1, False), (8, 150, 2, False), (32, 300, 2, True), (16, 5, 1, False)))
def test_pool_forward_then_inverse_equals_step(pq, m, S, C, downmix):
    mod = pq.CachedPQMF(100, m).cuda()
    rows = S * (1 if downmix else C)
    a, b = pq.StreamPool(mod, rows + 3), pq.StreamPool(mod, rows + 3)
    for k in range(3):
        ids = torch.randperm(rows + 3, device="cuda")[:rows].to(torch.int32)
        pcm = pcm_blocks((S, 2048 if k != 1 else 3 * m, C), k + m)
        out_b, y_b = b.step_pcm16(pcm, ids, downmix)
        y_a = a.forward_pcm16(pcm, ids, downmix)
        out_a = a.inverse_pcm16(y_a, ids)
        assert torch.equal(y_a, y_b) and torch.equal(out_a, out_b), k
        for u, v in zip((a.xpool, a.spool, a.xphase, a.sphase), (b.xpool, b.spool, b.xphase, b.sphase)):
            assert torch.equal(u, v), k


@pytest.mark.gpu
@pytest.mark.parametrize("m,P,S,C,downmix", ((16, 900, 300, 1, False), (16, 900, 150, 2, True), (8, 40, 6, 1, False)))
def test_pool_graph_replays_any_ids(pq, m, P, S, C, downmix):
    """One captured step_pcm16 with CUDA ids replays with new ids and new blocks: bit-equal to an eager twin pool."""
    mod = pq.CachedPQMF(100, m).cuda()
    graph_pool, eager = pq.StreamPool(mod, P), pq.StreamPool(mod, P)
    rows = S * (1 if downmix else C)
    rng = np.random.default_rng(P + S)
    pre = torch.from_numpy(rng.choice(P, P // 3, replace=False).astype(np.int32)).cuda()  # mixed parities first, on both pools
    xpre = pcm_blocks((pre.numel(), 3 * m, 1), 9)
    graph_pool.step_pcm16(xpre, pre)
    eager.step_pcm16(xpre, pre)
    static_pcm = torch.zeros(S, 2048, C, dtype=torch.int16, device="cuda")
    static_ids = torch.arange(rows, dtype=torch.int32, device="cuda")
    warm = pq.StreamPool(mod, P)  # first launches set the kernels' shared-memory limits: not inside a capture
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        warm.step_pcm16(static_pcm, static_ids, downmix)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        g_out, g_y = graph_pool.step_pcm16(static_pcm, static_ids, downmix)
    for k in range(5):
        ids = torch.from_numpy(rng.choice(P, rows, replace=False).astype(np.int32)).cuda()
        pcm = pcm_blocks((S, 2048, C), 50 + k)
        static_pcm.copy_(pcm)
        static_ids.copy_(ids)
        graph.replay()
        out, y = eager.step_pcm16(pcm, ids, downmix)
        assert torch.equal(g_y, y) and torch.equal(g_out, out), k
        for u, v in zip((graph_pool.xpool, graph_pool.spool, graph_pool.xphase, graph_pool.sphase),
                        (eager.xpool, eager.spool, eager.xphase, eager.sphase)):
            assert torch.equal(u, v), k


@pytest.mark.gpu
@pytest.mark.parametrize("m,S,C,downmix", ((16, 300, 1, False), (8, 300, 2, True), (32, 300, 1, False)))
def test_streamed_equals_offline(pq, m, S, C, downmix):
    """A clip streamed through process_stream_pcm16 equals the offline forward_pcm16 / inverse_pcm16 on the zero-prefixed clip at the fixed
    latency: sub-bands within the fp32 tolerance, output within 1 LSB; sub-band excerpts also match the float64 oracle."""
    n_blocks, block = 4, 2048
    mod = pq.CachedPQMF(100, m).cuda()
    length = mod.hk.shape[1]
    t = n_blocks * block
    pcm = pcm_blocks((S, t, C), 11 + m)
    ys, outs = [], []
    for k in range(n_blocks):
        out, y = mod.process_stream_pcm16(pcm[:, k * block : (k + 1) * block].contiguous(), downmix)
        ys.append(y)
        outs.append(out)
    y_s, out_s = torch.cat(ys, -1), torch.cat(outs, 1)
    pz = torch.cat([torch.zeros(S, length // 2, C, dtype=torch.int16, device="cuda"), pcm], dim=1)
    y_off = mod.forward_pcm16(pz, downmix)[..., : t // m]
    assert (y_s - y_off).abs().max().item() <= 2e-6
    sz = torch.cat([torch.zeros(S, y_s.shape[1], (length // m) // 2, device="cuda"), y_s], dim=-1)
    o_off = mod.inverse_pcm16(sz)[:, :t]
    assert (out_s.int() - o_off.int()).abs().max().item() <= 1
    hk = mod.hk.cpu().double().numpy()
    x64 = widen(pcm, downmix).reshape(-1, t)[:3].cpu().double().numpy()
    st = O.StreamState(3, m, length)
    y64 = O.stream_analysis(x64, hk, st)
    assert np.abs(y_s.reshape(-1, m, t // m)[:3].cpu().numpy() - y64).max() <= 5e-6


@pytest.mark.gpu
def test_errors(pq):
    mod = pq.CachedPQMF(100, 16).cuda()
    pool = pq.StreamPool(mod, 16)
    with pytest.raises(RuntimeError, match="int16"):
        mod.forward_stream_pcm16(torch.zeros(3, 256, 1, device="cuda"))
    with pytest.raises(RuntimeError, match="int16"):
        pool.step_pcm16(torch.zeros(3, 256, 1, device="cuda"), [0, 1, 2])
    for dt, name in ((torch.float16, "Half"), (torch.bfloat16, "BFloat16")):
        with pytest.raises(RuntimeError, match=name):
            mod.inverse_stream_pcm16(torch.zeros(3, 16, 16, device="cuda", dtype=dt))
        with pytest.raises(RuntimeError, match=name):
            pool.inverse_pcm16(torch.zeros(3, 16, 16, device="cuda", dtype=dt), [0, 1, 2])
    with pytest.raises(RuntimeError):
        mod.forward_stream_pcm16(torch.zeros(3, 256, dtype=torch.int16, device="cuda"))  # wrong rank
    with pytest.raises(RuntimeError):
        mod.process_stream_pcm16(torch.zeros(3, 256, dtype=torch.int16, device="cuda"))
    with pytest.raises(RuntimeError):
        mod.inverse_stream_pcm16(torch.zeros(3, 16, device="cuda"))
    with pytest.raises(RuntimeError, match="ids has 3 entries"):
        pool.step_pcm16(torch.zeros(3, 256, 2, dtype=torch.int16, device="cuda"), torch.tensor([0, 1, 2], device="cuda"))  # 6 rows
    with pytest.raises(RuntimeError, match="not differentiable"):
        mod.inverse_stream_pcm16(torch.zeros(3, 16, 16, device="cuda", requires_grad=True))
    with pytest.raises(RuntimeError, match="not differentiable"):
        pool.inverse_pcm16(torch.zeros(3, 16, 16, device="cuda", requires_grad=True), [0, 1, 2])
    with pytest.raises((RuntimeError, NotImplementedError)):
        torch.ops.pqmf_b200.analysis_stream_pcm16(torch.zeros(3, 256, 1, dtype=torch.int16), mod.hk.cpu(), mod._tables.cpu(), torch.zeros(3, 512),
                                                  torch.zeros(3, 512), 0, False, 0)
    with pytest.raises(RuntimeError):
        mod.forward_stream_pcm16(torch.zeros(3, 256, 1, dtype=torch.int16))  # CPU block, CUDA module
    assert (pool.xphase == 0).all() and (pool.sphase == 0).all()


def test_cabi_argument_checks_happen_before_any_cuda_call(pq):
    """The six PCM streaming entries validate on the host and return PQMF_ERR_ARG (or 0 for no rows) without touching a device."""
    c = _cabi(pq)
    an, sy, st = c.pqmf_analysis_stream_pcm16, c.pqmf_synthesis_stream_pcm16, c.pqmf_stream_step_pcm16
    pa, ps, pst = c.pqmf_stream_pool_analysis_pcm16, c.pqmf_stream_pool_synthesis_pcm16, c.pqmf_stream_pool_step_pcm16
    n6, n9 = [None] * 6, [None] * 9
    # null pointers
    assert an(*n6, 4, 2048, 1, 0, 16, 512, 0, 0, None) == ERR_ARG
    assert sy(*n6, 4, 1, 128, 16, 512, 0, 0, None) == ERR_ARG
    assert st(*n9, 4, 2048, 1, 0, 16, 512, 0, 0, 0, None) == ERR_ARG
    assert pa(*n6, 8, None, 4, 2048, 1, 0, 16, 512, 0, None) == ERR_ARG
    assert ps(*n6, 8, None, 4, 1, 128, 16, 512, 0, None) == ERR_ARG
    assert pst(*n9, 8, None, 4, 2048, 1, 0, 16, 512, 0, None) == ERR_ARG
    # C < 1 (and C > 64)
    for C in (0, 65):
        assert an(*n6, 4, 2048, C, 0, 16, 512, 0, 0, None) == ERR_ARG
        assert sy(*n6, 4, C, 128, 16, 512, 0, 0, None) == ERR_ARG
        assert st(*n9, 4, 2048, C, 0, 16, 512, 0, 0, 0, None) == ERR_ARG
        assert pa(*n6, 8, None, 4, 2048, C, 0, 16, 512, 0, None) == ERR_ARG
        assert ps(*n6, 8, None, 4, C, 128, 16, 512, 0, None) == ERR_ARG
        assert pst(*n9, 8, None, 4, 2048, C, 0, 16, 512, 0, None) == ERR_ARG
    # T % M != 0
    assert an(*n6, 4, 2049, 1, 0, 16, 512, 0, 0, None) == ERR_ARG
    assert st(*n9, 4, 2049, 1, 0, 16, 512, 0, 0, 0, None) == ERR_ARG
    assert pa(*n6, 8, None, 4, 2049, 1, 0, 16, 512, 0, None) == ERR_ARG
    assert pst(*n9, 8, None, 4, 2049, 1, 0, 16, 512, 0, None) == ERR_ARG
    # more rows than streams in the pool: 3 stereo blocks are 6 rows
    assert pa(*n6, 5, None, 3, 2048, 2, 0, 16, 512, 0, None) == ERR_ARG
    assert ps(*n6, 5, None, 3, 2, 128, 16, 512, 0, None) == ERR_ARG
    assert pst(*n9, 5, None, 3, 2048, 2, 0, 16, 512, 0, None) == ERR_ARG
    # no rows: nothing to do
    assert an(*n6, 0, 2048, 1, 0, 16, 512, 0, 0, None) == 0
    assert sy(*n6, 0, 1, 128, 16, 512, 0, 0, None) == 0
    assert st(*n9, 0, 2048, 1, 0, 16, 512, 0, 0, 0, None) == 0
    assert pa(*n6, 8, None, 0, 2048, 1, 0, 16, 512, 0, None) == 0
    assert ps(*n6, 8, None, 0, 1, 128, 16, 512, 0, None) == 0
    assert pst(*n9, 8, None, 0, 2048, 1, 0, 16, 512, 0, None) == 0
