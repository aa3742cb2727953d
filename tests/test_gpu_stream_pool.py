"""Stream pools: P independent streams with device-resident state, any subset of which one call steps, in any order.

Per row, a pool call must give the bits of the lockstep streaming entries run on that stream's own state and parity, on the same kernel
family (the streaming Hankel-4 kernels where a lockstep call with as many rows runs them, the direct form elsewhere); streams that are
not listed must be left untouched, bit for bit.  The last test needs no GPU: it checks the C entries' argument validation."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import pqmf_oracle as O

TOL = 1e-5
FP32 = 16  # PQMF_FLAG_FP32
# n_band 16 / L 512, 2048-sample blocks: 3 streams per MMA tile, and the Hankel-4 kernels take >= 96 tiles = 286 streams
H4_MIN_STREAMS = 286


@pytest.fixture(scope="module")
def pq():
    import pqmf_b200

    return pqmf_b200


def _blocks(streams, block, n_blocks, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (0.5 * torch.randn(n_blocks, streams, 1, block, device="cuda", generator=g)).clamp_(-1, 1)


@pytest.mark.gpu
@pytest.mark.parametrize("m,streams,block,fp32_ref", (
    (16, 300, 2048, False), (16, 4096, 2048, False), (8, 1000, 512, False), (32, 290, 4096, False),  # Hankel-4 family
    (8, 7, 2048, False), (32, 5, 1024, False), (64, 2, 4096, False), (4, 3, 256, False),             # direct form
    (16, 7, 2048, True)))                                                                              # direct form on both sides
def test_lockstep_ids_equal_process_stream(pq, m, streams, block, fp32_ref):
    """ids = arange(S) every block: outputs, both states and the phase words equal CachedPQMF.process_stream, bit for bit."""
    mod = pq.CachedPQMF(100, m).cuda()
    ref = pq.CachedPQMF(100, m, fp32=fp32_ref).cuda()
    assert torch.equal(mod.hk, ref.hk)
    pool = pq.StreamPool(mod, streams)
    ids = torch.arange(streams, device="cuda", dtype=torch.int32)
    xs = _blocks(streams, block, 5, m * streams + block)
    for k in range(xs.shape[0]):
        out, y = pool.step(xs[k], ids)
        out_r, y_r = ref.process_stream(xs[k])
        assert torch.equal(y, y_r) and torch.equal(out, out_r), k
        assert torch.equal(pool.xpool, ref._x_state) and torch.equal(pool.spool.reshape(2, streams, -1), ref._s_state), k
        word = ((k + 1) & 1) | ((((k + 1) * (block // m)) & 1) << 1)
        assert (pool.xphase == word).all() and (pool.sphase == word).all()


def _lockstep_reference(pq, mod, x, ids, xpool, spool, xphase, sphase, h4):
    """What the lockstep stream_step gives each listed stream on its own gathered state, grouped by parity; Hankel-4 groups padded with
    zero streams up to the kernels' tile threshold, direct-form groups forced there with PQMF_FLAG_FP32."""
    n, T = x.shape[0], x.shape[-1]
    y = torch.empty(n, mod.n_band, T // mod.n_band, device="cuda")
    out = torch.empty(n, 1, T, device="cuda")
    xnew = torch.empty(n, xpool.shape[-1], device="cuda")
    snew = torch.empty(n, spool[0, 0].numel(), device="cuda")
    idl = ids.long()
    xh, sh = xphase[idl] & 1, sphase[idl] & 1
    px, ps = (xphase[idl] >> 1) & 1, (sphase[idl] >> 1) & 1
    rows = torch.arange(n, device="cuda")
    for a in (0, 1):
        for b in (0, 1):
            sel = rows[(px == a) & (ps == b)]
            if sel.numel() == 0:
                continue
            g = sel.numel()
            pad = max(H4_MIN_STREAMS + 2 - g, 0) if h4 else 0
            def padded(t):
                return torch.cat([t, t.new_zeros((pad,) + tuple(t.shape[1:]))]) if pad else t.contiguous()
            xg = padded(x[sel])
            xs_in = padded(xpool[xh[sel], idl[sel]])
            ss_in = padded(spool[sh[sel], idl[sel]].reshape(g, -1))
            xs_out, ss_out = torch.empty_like(xs_in), torch.empty_like(ss_in)
            flags = mod._flags if h4 else mod._flags | FP32
            o, yy = torch.ops.pqmf_b200.stream_step(xg, mod.hk.float(), mod._tables, xs_in, xs_out, ss_in, ss_out, a, b, flags)
            y[sel], out[sel], xnew[sel], snew[sel] = yy[:g], o[:g], xs_out[:g], ss_out[:g]
    return out, y, xnew, snew


@pytest.mark.gpu
def test_independent_sessions(pq):
    """A seeded schedule over a pool of 4096: random subsets in random order, on both kernel families, 3-frame blocks that mix the
    parities, resets in the middle.  After every step: (a) every row and new state row equals the lockstep entry on that stream's own
    state, (b) streams not stepped keep both halves and their phase words, (c) sampled streams match the float64 oracle."""
    P, m, length = 4096, 16, 512
    mod = pq.CachedPQMF(100, m).cuda()
    pool = pq.StreamPool(mod, P)
    hk = mod.hk.cpu().double().numpy()
    rng = np.random.default_rng(2024)
    sample = [int(i) for i in rng.choice(P, 6, replace=False)]
    oracle = {i: O.StreamState(1, m, length) for i in sample}
    schedule = [(4096, 2048), (300, 2048), (150, 2048), (2000, 48), (3000, 2048), (90, 48), ("reset", 0), (500, 2048), (40, 2048),
                (4096, 48), (1200, 2048), (7, 2048), (2500, 2048)]
    for step, (n, T) in enumerate(schedule):
        if n == "reset":
            gone = sorted(set(rng.choice(P, 600, replace=False).tolist()) | set(sample[:2]))
            pool.reset(gone)
            for i in set(gone) & set(sample):
                oracle[i] = O.StreamState(1, m, length)
            assert pool.xpool[:, gone].abs().sum().item() == 0 and pool.spool[:, gone].abs().sum().item() == 0
            assert (pool.xphase[gone] == 0).all() and (pool.sphase[gone] == 0).all()
            continue
        inc = rng.choice(sample, min(3, n), replace=False)  # some sampled streams in every step, the others when drawn
        others = rng.choice(np.setdiff1d(np.arange(P), inc), n - len(inc), replace=False)
        chosen = rng.permutation(np.concatenate([inc, others]))
        ids = torch.from_numpy(chosen.astype(np.int32)).cuda()
        x = (0.5 * torch.randn(n, 1, T, device="cuda")).clamp_(-1, 1)
        before = [t.clone() for t in (pool.xpool, pool.spool, pool.xphase, pool.sphase)]
        h4 = T % 256 == 0 and n >= H4_MIN_STREAMS
        out_r, y_r, xnew_r, snew_r = _lockstep_reference(pq, mod, x, ids, *before, h4)
        out, y = pool.step(x, ids)
        assert torch.equal(y, y_r) and torch.equal(out, out_r), step
        idl = ids.long()
        assert torch.equal(pool.xpool[pool.xphase[idl].long() & 1, idl], xnew_r), step
        assert torch.equal(pool.spool[pool.sphase[idl].long() & 1, idl].reshape(n, -1), snew_r), step
        frames = T // m
        assert torch.equal(pool.xphase[idl], (before[2][idl] ^ 1) & 1 | ((((before[2][idl] >> 1) + frames) & 1) << 1))
        assert torch.equal(pool.sphase[idl], pool.xphase[idl])
        # (b) untouched streams
        rest = torch.ones(P, dtype=torch.bool, device="cuda")
        rest[idl] = False
        assert torch.equal(pool.xpool[:, rest], before[0][:, rest]) and torch.equal(pool.spool[:, rest], before[1][:, rest]), step
        assert torch.equal(pool.xphase[rest], before[2][rest]) and torch.equal(pool.sphase[rest], before[3][rest]), step
        # (c) the oracle, per sampled stream, counting frames from its last reset
        pos = {int(v): r for r, v in enumerate(chosen)}
        for i in sample:
            if i in pos:
                st, r = oracle[i], pos[i]
                y64 = O.stream_analysis(x[r : r + 1, 0].cpu().double().numpy(), hk, st)
                o64 = O.stream_synthesis(y[r : r + 1].cpu().double().numpy(), hk, st)
                assert np.abs(y[r : r + 1].cpu().numpy() - y64).max() <= TOL / 2, (step, i)
                assert np.abs(out[r : r + 1, 0].cpu().numpy() - o64).max() <= TOL / 2, (step, i)


@pytest.mark.gpu
def test_forward_then_inverse_equals_step_and_directions_keep_their_parity(pq):
    m, S = 8, 5
    mod = pq.CachedPQMF(100, m).cuda()
    a, b = pq.StreamPool(mod, S), pq.StreamPool(mod, S)
    xs = _blocks(S, 2048, 3, 5)
    for k in range(3):
        ids = torch.randperm(S, device="cuda").to(torch.int32)
        out_b, y_b = b.step(xs[k], ids)
        y_a = a.forward(xs[k], ids)
        out_a = a.inverse(y_a, ids)
        assert torch.equal(y_a, y_b) and torch.equal(out_a, out_b)
        for u, v in zip((a.xpool, a.spool, a.xphase, a.sphase), (b.xpool, b.spool, b.xphase, b.sphase)):
            assert torch.equal(u, v)
    # uneven directions: 3-frame analysis blocks ahead of the synthesis, against forward_stream / inverse_stream of a lockstep module
    pool, ref = pq.StreamPool(mod, S), pq.CachedPQMF(100, m).cuda()
    x3f = _blocks(S, 24, 4, 6)  # 3 frames per block
    order = [torch.randperm(S, device="cuda") for _ in range(4)]
    ys = []
    for k in range(2):
        y = pool.forward(x3f[k][order[k]], order[k].to(torch.int32))
        y_r = ref.forward_stream(x3f[k])
        assert torch.equal(y, y_r[order[k]])
        ys.append(y_r)
    assert ((pool.xphase >> 1) == 0).all() and ((pool.sphase >> 1) == 0).all() and (pool.xphase == 0).all()  # 6 frames: even again
    for k in range(2, 4):
        y = pool.forward(x3f[k][order[k]], order[k].to(torch.int32))
        y_r = ref.forward_stream(x3f[k])
        assert torch.equal(y, y_r[order[k]])
        ys.append(y_r)
        out = pool.inverse(ys[k - 2][order[k]], order[k].to(torch.int32))
        assert torch.equal(out, ref.inverse_stream(ys[k - 2])[order[k]])
        assert ((pool.sphase >> 1) & 1).tolist() == [(3 * (k - 1)) & 1] * S and ((pool.xphase >> 1) & 1).tolist() == [(3 * (k + 1)) & 1] * S


@pytest.mark.gpu
@pytest.mark.parametrize("m,P,n,block", ((16, 900, 300, 2048), (16, 12, 5, 48), (8, 40, 6, 2048)))
def test_one_graph_replays_any_ids_and_frame_counts(pq, m, P, n, block):
    """One captured pool step replays with new ids and new blocks; the parities live on the device, so odd frame counts per block
    need no second graph.  Bit-equal to an eager twin pool."""
    mod = pq.CachedPQMF(100, m).cuda()
    graph_pool, eager = pq.StreamPool(mod, P), pq.StreamPool(mod, P)
    rng = np.random.default_rng(P + block)
    # mix the parities first (3-frame blocks on some streams, direct form), identically on both pools
    pre = torch.from_numpy(rng.choice(P, P // 3, replace=False).astype(np.int32)).cuda()
    xpre = (0.5 * torch.randn(pre.numel(), 1, 3 * m, device="cuda")).clamp_(-1, 1)
    graph_pool.step(xpre, pre)
    eager.step(xpre, pre)
    static_x = torch.zeros(n, 1, block, device="cuda")
    static_ids = torch.arange(n, dtype=torch.int32, device="cuda")
    warm = pq.StreamPool(mod, P)  # first launches set the kernels' shared-memory limits: not inside a capture
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        warm.step(static_x, static_ids)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        g_out, g_y = graph_pool.step(static_x, static_ids)
    for k in range(6):
        ids = torch.from_numpy(rng.choice(P, n, replace=False).astype(np.int32)).cuda()
        x = (0.5 * torch.randn(n, 1, block, device="cuda")).clamp_(-1, 1)
        static_x.copy_(x)
        static_ids.copy_(ids)
        graph.replay()
        out, y = eager.step(x, ids)
        assert torch.equal(g_y, y) and torch.equal(g_out, out), k
        for u, v in zip((graph_pool.xpool, graph_pool.spool, graph_pool.xphase, graph_pool.sphase), (eager.xpool, eager.spool, eager.xphase, eager.sphase)):
            assert torch.equal(u, v), k


@pytest.mark.gpu
@pytest.mark.parametrize("m,streams,block", ((16, 7, 2048), (16, 300, 2048), (8, 5, 256)))
def test_streamed_equals_offline_out_of_order(pq, m, streams, block):
    """Each stream of a pool stepped in random subsets and orders: its concatenated sub-bands and signal satisfy the zero-prefixed
    offline invariants of test_gpu_streaming.test_streamed_equals_offline."""
    n_blocks = 5
    mod = pq.CachedPQMF(100, m).cuda()
    length = mod.hk.shape[1]
    pool = pq.StreamPool(mod, streams)
    x = torch.from_numpy(O.audio_like((streams, 1, n_blocks * block), 31 + block)).cuda()
    y_s = torch.zeros(streams, m, n_blocks * block // m, device="cuda")
    out_s = torch.zeros(streams, 1, n_blocks * block, device="cuda")
    done = np.zeros(streams, int)
    rng = np.random.default_rng(streams)
    while (done < n_blocks).any():
        left = np.flatnonzero(done < n_blocks)
        pick = rng.permutation(left)[: max(1, int(rng.integers(len(left) // 2, len(left) + 1)))]
        blk = [slice(int(done[i]) * block, int(done[i] + 1) * block) for i in pick]
        xb = torch.stack([x[i, :, s] for i, s in zip(pick, blk)])
        out, y = pool.step(xb, pick.tolist())
        for r, (i, s) in enumerate(zip(pick, blk)):
            y_s[i, :, s.start // m : s.stop // m] = y[r]
            out_s[i, :, s] = out[r]
        done[pick] += 1
    t = n_blocks * block
    xz = torch.cat([torch.zeros(streams, 1, length // 2, device="cuda"), x], dim=-1)
    assert (y_s - mod.forward(xz)[..., : t // m]).abs().max().item() <= 2e-6
    sz = torch.cat([torch.zeros(streams, m, (length // m) // 2, device="cuda"), y_s], dim=-1)
    assert (out_s - mod.inverse(sz)[..., :t]).abs().max().item() <= 4e-6


@pytest.mark.gpu
def test_pool_errors(pq):
    mod = pq.CachedPQMF(100, 16).cuda()
    pool = pq.StreamPool(mod, 8)
    x = torch.zeros(3, 1, 256, device="cuda")
    launches = pq.launch_count()
    for bad in ([0, 1, 1], [0, 1, 8], [-1, 2, 3], torch.tensor([0, 0, 2])):
        with pytest.raises(ValueError):
            pool.step(x, bad)
    assert pq.launch_count() == launches and (pool.xphase == 0).all()
    with pytest.raises(RuntimeError):
        pool.step(x, torch.tensor([0, 1], device="cuda"))      # 3 rows, 2 ids
    with pytest.raises(RuntimeError):
        pool.step(x[:, 0], torch.tensor([0, 1, 2], device="cuda"))  # wrong rank
    with pytest.raises(RuntimeError):
        pool.inverse(torch.zeros(3, 8, 16, device="cuda"), [0, 1, 2])  # not n_band channels
    for dt, name in ((torch.float16, "Half"), (torch.bfloat16, "BFloat16")):
        with pytest.raises(RuntimeError, match=name):
            pool.step(x.to(dt), [0, 1, 2])
        with pytest.raises(RuntimeError, match=name):
            pool.inverse(torch.zeros(3, 16, 16, device="cuda", dtype=dt), [0, 1, 2])
    with pytest.raises(RuntimeError, match="not differentiable"):
        pool.step(x.clone().requires_grad_(), [0, 1, 2])
    with pytest.raises(RuntimeError, match="not differentiable"):
        pool.forward(x.clone().requires_grad_(), [0, 1, 2])
    with pytest.raises(RuntimeError, match="not differentiable"):
        pool.inverse(torch.zeros(3, 16, 16, device="cuda", requires_grad=True), [0, 1, 2])
    assert (pool.xphase == 0).all() and (pool.sphase == 0).all()


def test_pool_cabi_argument_checks_happen_before_any_cuda_call(pq):
    """The pool entries validate on the host and return PQMF_ERR_ARG (or 0 for n == 0) without touching a device: runs on a CPU box."""
    c = pq._lib.cabi
    vp, i, lg, u = ctypes.c_void_p, ctypes.c_int, ctypes.c_long, ctypes.c_uint
    c.pqmf_stream_pool_analysis_f32.argtypes = [vp] * 6 + [i, vp, i, lg, i, i, u, vp]
    c.pqmf_stream_pool_synthesis_f32.argtypes = [vp] * 6 + [i, vp, i, lg, i, i, u, vp]
    c.pqmf_stream_pool_step_f32.argtypes = [vp] * 9 + [i, vp, i, lg, i, i, u, vp]
    for f in (c.pqmf_stream_pool_analysis_f32, c.pqmf_stream_pool_synthesis_f32, c.pqmf_stream_pool_step_f32):
        f.restype = ctypes.c_int
    an, sy, st = c.pqmf_stream_pool_analysis_f32, c.pqmf_stream_pool_synthesis_f32, c.pqmf_stream_pool_step_f32
    nul6, nul9 = [None] * 6, [None] * 9
    # null pointers
    assert an(*nul6, 8, None, 4, 2048, 16, 512, 0, None) == -1
    assert sy(*nul6, 8, None, 4, 128, 16, 512, 0, None) == -1
    assert st(*nul9, 8, None, 4, 2048, 16, 512, 0, None) == -1
    # n > P
    assert an(*nul6, 4, None, 5, 2048, 16, 512, 0, None) == -1
    assert sy(*nul6, 4, None, 5, 128, 16, 512, 0, None) == -1
    assert st(*nul9, 4, None, 5, 2048, 16, 512, 0, None) == -1
    # T % M != 0
    assert an(*nul6, 8, None, 0, 2049, 16, 512, 0, None) == -1
    assert st(*nul9, 8, None, 0, 2049, 16, 512, 0, None) == -1
    # P < 1
    assert an(*nul6, 0, None, 0, 2048, 16, 512, 0, None) == -1
    assert sy(*nul6, 0, None, 0, 128, 16, 512, 0, None) == -1
    assert st(*nul9, 0, None, 0, 2048, 16, 512, 0, None) == -1
    # n == 0: nothing to do
    assert an(*nul6, 8, None, 0, 2048, 16, 512, 0, None) == 0
    assert sy(*nul6, 8, None, 0, 128, 16, 512, 0, None) == 0
    assert st(*nul9, 8, None, 0, 2048, 16, 512, 0, None) == 0
