"""Grouped stream-pool calls: sessions of different block lengths stepped in one call (StreamPool.step_groups / forward_groups /
inverse_groups, pqmf_stream_pool_*_groups_f32).

The routing rule: the groups the streaming Hankel-4 kernels can plan (family, block geometry, flags, alignment -- whatever their own tile
count) run together in one GROUPS launch per direction plus one phase-word launch, when there are at least two of them and they make >= 96
tiles together; every other group runs through its single-group pool entry.  So a grouped row equals the same stream stepped by a
single-group call that runs the streaming Hankel-4 kernels (padded with zero streams of a scratch pool when the group alone is too small),
and a fallback row equals `step` of its own group.  The last test needs no GPU: it checks the C entries' argument validation."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import pqmf_oracle as O

TOL = 1e-5
MIN_TILES = 96
FLAG_BLOCKERS = 2 | 4 | 8 | 16 | (1 << 23)  # NO_SIGN, FOLD, NO_PAIR, FP32, H4_SPLIT


@pytest.fixture(scope="module")
def pq():
    import pqmf_b200

    return pqmf_b200


def _geom(rows_b, hist):
    hrows = hist // 64
    pitch = (rows_b + hrows + 3) & ~3
    return pitch, 128 // pitch


def _spt(mod, T):
    """Streams per tile of a block of T samples in each direction (h4_*_stream_plan), or None where the streaming Hankel-4 kernels
    cannot plan the block whatever the number of streams."""
    m, length = mod.hk.shape
    flags = mod._flags
    jlo, kt = 32 * ((flags >> 8) & 0xF), 32 * ((flags >> 12) & 0x1F)
    if m not in (8, 16, 32) or mod._tables.numel() == 0 or kt == 0 or flags & FLAG_BLOCKERS:
        return None
    hist_a = -(-(length - jlo) // 64) * 64
    taps = (jlo + kt) // m
    hist_fr = -(-(taps * m) // 64) * 64 // m
    F, K = T // m, length // m
    if hist_a > length or T % 256 or T < length or length % 8:
        return None
    if hist_fr % 4 or hist_fr > K or (F * m) % 256 or F % 4 or F < K:
        return None
    pa, sa = _geom(T // 64, hist_a)
    ps, ss = _geom(T // 64, hist_fr * m)
    if pa > 128 or ps > 128 or sa < 1 or ss < 1:
        return None
    return sa, ss


def _tiles(n, spt):
    return -(-n // spt)


def _joined(mod, shapes, aligned=None):
    """Indices of the groups (n, T) that run in the grouped launch of a step."""
    if len(shapes) < 2:
        return set()
    plan = {}
    for k, (n, T) in enumerate(shapes):
        s = _spt(mod, T)
        if n > 0 and s is not None and (aligned is None or aligned[k]):
            plan[k] = s
    ta = sum(_tiles(shapes[k][0], s[0]) for k, s in plan.items())
    ts = sum(_tiles(shapes[k][0], s[1]) for k, s in plan.items())
    return set(plan) if len(plan) >= 2 and ta >= MIN_TILES and ts >= MIN_TILES else set()


def _blocks(n, T, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (0.5 * torch.randn(n, 1, T, device="cuda", generator=g)).clamp_(-1, 1)


def _state(pool):
    return [t.clone() for t in (pool.xpool, pool.spool, pool.xphase, pool.sphase)]


def _assert_pools_equal(a, b, what=""):
    for u, v in zip((a.xpool, a.spool, a.xphase, a.sphase), (b.xpool, b.spool, b.xphase, b.sphase)):
        assert torch.equal(u, v), what


def _padded_step(pq, mod, pool, x, ids):
    """`step` of the rows (x, ids) of `pool` on the streaming Hankel-4 kernels: the streams' state and phase words copied into a scratch pool
    padded with zero streams up to the tile threshold, one single-T step there, the new state and words copied back into `pool`."""
    n, T = x.shape[0], x.shape[-1]
    sa, ss = _spt(mod, T)
    cap = max(n, MIN_TILES * max(sa, ss))
    idl = ids.long()
    s = pq.StreamPool(mod, cap)
    s.xpool[:, :n], s.spool[:, :n] = pool.xpool[:, idl], pool.spool[:, idl]
    s.xphase[:n], s.sphase[:n] = pool.xphase[idl], pool.sphase[idl]
    out, y = s.step(torch.cat([x, x.new_zeros(cap - n, 1, T)]), torch.arange(cap, dtype=torch.int32, device="cuda"))
    pool.xpool[:, idl], pool.spool[:, idl] = s.xpool[:, :n], s.spool[:, :n]
    pool.xphase[idl], pool.sphase[idl] = s.xphase[:n], s.sphase[:n]
    return out[:n], y[:n]


def _reference_step(pq, mod, twin, groups, joined):
    """What step_groups must give, group by group, on the twin pool."""
    res = []
    for k, (x, ids) in enumerate(groups):
        res.append(_padded_step(pq, mod, twin, x, ids) if k in joined else twin.step(x, ids))
    return res


def _check_oracle(mod, before, x, y, out, ids, rows, what):
    m, length = mod.hk.shape
    hk = mod.hk.cpu().double().numpy()
    xpool, spool, xphase, sphase = before
    for r in rows:
        i = int(ids[r])
        st = O.StreamState(1, m, length)
        st.x_hist = xpool[int(xphase[i]) & 1, i].cpu().double().numpy()[None]
        st.s_hist = spool[int(sphase[i]) & 1, i].cpu().double().numpy()[None]
        st.frames_in, st.frames_out = (int(xphase[i]) >> 1) & 1, (int(sphase[i]) >> 1) & 1
        y64 = O.stream_analysis(x[r : r + 1, 0].cpu().double().numpy(), hk, st)
        o64 = O.stream_synthesis(y[r : r + 1].cpu().double().numpy(), hk, st)
        assert np.abs(y[r : r + 1].cpu().numpy() - y64).max() <= TOL / 2, (what, r)
        assert np.abs(out[r : r + 1, 0].cpu().numpy() - o64).max() <= TOL / 2, (what, r)


# n_band -> block lengths whose groups are each >= 96 tiles alone (the largest native block at n_band 16 / attenuation 100: 7680 samples =
# 120 block rows + 7 history rows, one stream per tile)
NATIVE = {8: (512, 1024, 2048), 16: (512, 2048, 7680), 32: (1024, 2048, 4096)}


@pytest.mark.gpu
@pytest.mark.parametrize("m", (8, 16, 32))
def test_native_groups_equal_sequential_steps(pq, m):
    mod = pq.CachedPQMF(100, m).cuda()
    shapes = []
    for T in NATIVE[m]:
        s = _spt(mod, T)
        assert s is not None, (m, T)
        shapes.append((MIN_TILES * max(s) + 5, T))
    P = sum(n for n, _ in shapes) + 64
    a, b = pq.StreamPool(mod, P), pq.StreamPool(mod, P)
    perm = torch.randperm(P, device="cuda").to(torch.int32)
    ids, r0 = [], 0
    for n, _ in shapes:
        ids.append(perm[r0 : r0 + n])
        r0 += n
    for step in range(3):
        groups = [(_blocks(n, T, 100 * step + k), ids[k]) for k, (n, T) in enumerate(shapes)]
        launches = pq.launch_count()
        got = a.step_groups(groups)
        assert pq.launch_count() - launches == 3
        launches = pq.launch_count()
        want = [b.step(x, i) for x, i in groups]
        assert pq.launch_count() - launches == 3 * len(groups)
        for (o, y), (o_r, y_r) in zip(got, want):
            assert torch.equal(y, y_r) and torch.equal(o, o_r), step
        _assert_pools_equal(a, b, step)
    # one direction at a time
    groups = [(_blocks(n, T, 7 + k), ids[k]) for k, (n, T) in enumerate(shapes)]
    launches = pq.launch_count()
    ys = a.forward_groups(groups)
    assert pq.launch_count() - launches == 2
    for y, (x, i) in zip(ys, groups):
        assert torch.equal(y, b.forward(x, i))
    launches = pq.launch_count()
    outs = a.inverse_groups([(y, i) for y, (_, i) in zip(ys, groups)])
    assert pq.launch_count() - launches == 2
    for o, y, (_, i) in zip(outs, ys, groups):
        assert torch.equal(o, b.inverse(y, i))
    _assert_pools_equal(a, b)


SERVER_MIX = ((600, 512), (400, 1024), (250, 2048), (90, 4096))  # n_band 16: 75 + 80 + 84 + 90 tiles, each below 96 alone


@pytest.mark.gpu
def test_small_groups_reach_the_tensor_cores_together(pq):
    mod = pq.CachedPQMF(100, 16).cuda()
    assert [_tiles(n, _spt(mod, T)[0]) for n, T in SERVER_MIX] == [75, 80, 84, 90]
    assert _joined(mod, SERVER_MIX) == {0, 1, 2, 3}
    P = 2048
    pool, twin, alone = pq.StreamPool(mod, P), pq.StreamPool(mod, P), pq.StreamPool(mod, P)
    perm = torch.randperm(P, device="cuda").to(torch.int32)
    ids, r0 = [], 0
    for n, _ in SERVER_MIX:
        ids.append(perm[r0 : r0 + n])
        r0 += n
    for step in range(2):
        groups = [(_blocks(n, T, 10 * step + k), ids[k]) for k, (n, T) in enumerate(SERVER_MIX)]
        before = _state(pool)
        launches = pq.launch_count()
        got = pool.step_groups(groups)
        assert pq.launch_count() - launches == 3
        want = _reference_step(pq, mod, twin, groups, {0, 1, 2, 3})
        direct = [alone.step(x, i) for x, i in groups]  # each group alone is below the threshold: the direct form
        for k, ((o, y), (o_r, y_r), (o_d, y_d)) in enumerate(zip(got, want, direct)):
            assert torch.equal(y, y_r) and torch.equal(o, o_r), (step, k)
            assert not torch.equal(y, y_d), (step, k)  # the route: not the direct form's bits
            n = o.shape[0]
            _check_oracle(mod, before, groups[k][0], y, o, ids[k], (0, n // 2, n - 1), (step, k))
        _assert_pools_equal(pool, twin, step)


@pytest.mark.gpu
def test_steady_state_across_group_boundaries(pq):
    """About ten tiles per CTA over four groups with different streams per tile, an odd tile count and a one-stream last tile in each
    group.  Each group alone is native, so the whole call equals sequential steps bit for bit; oracle rows on every CTA's first, second,
    third and last tile and on both sides of every group boundary."""
    mod = pq.CachedPQMF(100, 16).cuda()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    grid = sms & ~1
    per_group = (10 * grid) // 4 | 1  # odd
    shapes = []
    for T in (512, 1024, 2048, 4096):
        spt = _spt(mod, T)[0]
        shapes.append(((per_group - 1) * spt + 1, T))
    tiles = [per_group] * 4
    total = sum(tiles)
    P = sum(n for n, _ in shapes) + 17
    a, b = pq.StreamPool(mod, P), pq.StreamPool(mod, P)
    perm = torch.randperm(P, device="cuda").to(torch.int32)
    ids, r0 = [], 0
    for n, _ in shapes:
        ids.append(perm[r0 : r0 + n])
        r0 += n
    # tiles to check against the oracle: (group, first row, streams in the tile)
    tile0 = np.cumsum([0] + tiles)
    picks = set()
    for c in range(grid):
        its = list(range(c, total, grid))
        picks.update(its[:3] + its[-1:])
    for k in range(1, 4):
        picks.update((tile0[k] - 1, tile0[k]))
    for step in range(2):
        groups = [(_blocks(n, T, 50 + 10 * step + k), ids[k]) for k, (n, T) in enumerate(shapes)]
        before = _state(a)
        got = a.step_groups(groups)
        want = [b.step(x, i) for x, i in groups]
        for (o, y), (o_r, y_r) in zip(got, want):
            assert torch.equal(y, y_r) and torch.equal(o, o_r), step
        _assert_pools_equal(a, b, step)
        if step == 1:
            for t in sorted(picks):
                k = int(np.searchsorted(tile0, t, side="right") - 1)
                spt = _spt(mod, shapes[k][1])[0]
                row = (t - tile0[k]) * spt
                last = min(row + spt, shapes[k][0]) - 1
                x, i = groups[k]
                o, y = got[k]
                _check_oracle(mod, before, x, y, o, i, sorted({row, last}), (t, k))


@pytest.mark.gpu
def test_native_and_fallback_groups_in_one_call(pq):
    mod = pq.CachedPQMF(100, 16).cuda()
    P = 2048
    pool, twin = pq.StreamPool(mod, P), pq.StreamPool(mod, P)
    perm = torch.randperm(P, device="cuda").to(torch.int32)
    shapes = [(600, 512), (50, 48), (400, 1024), (40, 480), (300, 2048)]  # the last one misaligned
    ids, r0 = [], 0
    for n, _ in shapes:
        ids.append(perm[r0 : r0 + n])
        r0 += n
    aligned = [True, True, True, True, False]
    joined = _joined(mod, shapes, aligned)
    assert joined == {0, 2}
    for step in range(3):
        groups = []
        for k, (n, T) in enumerate(shapes):
            x = _blocks(n, T, 30 + 10 * step + k)
            if not aligned[k]:  # a contiguous view 4 bytes into its storage: refused by the streaming Hankel-4 kernels
                buf = torch.empty(n * T + 1, device="cuda")
                buf[1:].copy_(x.reshape(-1))
                x = buf[1:].view(n, 1, T)
                assert x.is_contiguous() and x.data_ptr() % 32 != 0
            groups.append((x, ids[k]))
        before = _state(pool)
        launches = pq.launch_count()
        got = pool.step_groups(groups)
        assert pq.launch_count() - launches == 3 + 3 * (len(shapes) - len(joined))
        want = _reference_step(pq, mod, twin, groups, joined)
        for k, ((o, y), (o_r, y_r)) in enumerate(zip(got, want)):
            assert torch.equal(y, y_r) and torch.equal(o, o_r), (step, k)
            _check_oracle(mod, before, groups[k][0], y, o, ids[k], (0, o.shape[0] - 1), (step, k))
        _assert_pools_equal(pool, twin, step)
    # n_band 4: every group falls back
    mod4 = pq.CachedPQMF(100, 4).cuda()
    p4, t4 = pq.StreamPool(mod4, 64), pq.StreamPool(mod4, 64)
    groups = [(_blocks(5, 256, 1), [0, 1, 2, 3, 4]), (_blocks(3, 512, 2), [10, 11, 12]), (_blocks(2, 64, 3), [20, 21])]
    launches = pq.launch_count()
    got = p4.step_groups(groups)
    assert pq.launch_count() - launches == 3 * len(groups)
    for (o, y), (x, i) in zip(got, groups):
        o_r, y_r = t4.step(x, i)
        assert torch.equal(y, y_r) and torch.equal(o, o_r)
    _assert_pools_equal(p4, t4)


@pytest.mark.gpu
def test_seeded_schedule_over_a_pool(pq):
    """Twelve steps over a pool of 4096: random subsets partitioned into random groups with random block lengths (mixing the parities),
    resets in between.  Against the twin pool (per the routing rule), the float64 oracle on sampled rows; streams not listed keep both
    halves and their phase words; a dead CUDA id gives zeros and touches no state."""
    P = 4096
    mod = pq.CachedPQMF(100, 16).cuda()
    pool, twin = pq.StreamPool(mod, P), pq.StreamPool(mod, P)
    rng = np.random.default_rng(7)
    lengths = (48, 256, 512, 1024, 2048, 4096)
    for step in range(12):
        if step in (4, 9):
            gone = rng.choice(P, 500, replace=False).tolist()
            pool.reset(gone)
            twin.reset(gone)
        G = int(rng.integers(2, 9))
        n_all = int(rng.integers(G, 3000))
        chosen = rng.choice(P, n_all, replace=False)
        cuts = np.sort(rng.choice(np.arange(1, n_all), G - 1, replace=False))
        parts = np.split(chosen, cuts)
        groups, shapes = [], []
        for k, part in enumerate(parts):
            T = int(rng.choice(lengths))
            groups.append((_blocks(len(part), T, 1000 * step + k), torch.from_numpy(part.astype(np.int32)).cuda()))
            shapes.append((len(part), T))
        dead = step == 6
        if dead:  # one dead row in the first group: ids outside [0, P)
            x0, i0 = groups[0]
            groups[0] = (x0, torch.cat([i0, torch.tensor([P + 3], dtype=torch.int32, device="cuda")]))
            groups[0] = (torch.cat([x0, _blocks(1, x0.shape[-1], 5)]), groups[0][1])
            shapes[0] = (shapes[0][0] + 1, shapes[0][1])
        joined = _joined(mod, shapes)
        before = _state(pool)
        got = pool.step_groups(groups)
        live = [(x[:-1], i[:-1]) if dead and k == 0 else (x, i) for k, (x, i) in enumerate(groups)]
        want = _reference_step(pq, mod, twin, live, joined)
        for k, ((o, y), (o_r, y_r)) in enumerate(zip(got, want)):
            n = o_r.shape[0]
            assert torch.equal(y[:n], y_r) and torch.equal(o[:n], o_r), (step, k)
            if dead and k == 0:
                assert (y[n:] == 0).all() and (o[n:] == 0).all()
        _assert_pools_equal(pool, twin, step)
        listed = torch.cat([i for _, i in live]).long()
        rest = torch.ones(P, dtype=torch.bool, device="cuda")
        rest[listed] = False
        for now, then in zip(_state(pool), before):
            assert torch.equal(now[:, rest] if now.dim() > 1 else now[rest], then[:, rest] if then.dim() > 1 else then[rest]), step
        for k in rng.choice(len(live), min(2, len(live)), replace=False):
            x, i = live[k]
            o, y = got[k]
            if x.shape[0]:
                _check_oracle(mod, before, x, y, o, i, (0, x.shape[0] - 1), (step, int(k)))


@pytest.mark.gpu
def test_one_graph_replays_grouped_steps(pq):
    mod = pq.CachedPQMF(100, 16).cuda()
    P = 2048
    graph_pool, eager = pq.StreamPool(mod, P), pq.StreamPool(mod, P)
    rng = np.random.default_rng(3)
    pre = torch.from_numpy(rng.choice(P, P // 3, replace=False).astype(np.int32)).cuda()  # mixed parities, identically on both pools
    xpre = (0.5 * torch.randn(pre.numel(), 1, 48, device="cuda")).clamp_(-1, 1)
    graph_pool.step(xpre, pre)
    eager.step(xpre, pre)
    static = [(torch.zeros(n, 1, T, device="cuda"), torch.arange(r0, r0 + n, dtype=torch.int32, device="cuda"))
              for (n, T), r0 in zip(SERVER_MIX, np.cumsum([0] + [n for n, _ in SERVER_MIX])[:-1].tolist())]
    warm = pq.StreamPool(mod, P)  # first launches set the kernels' shared-memory limits: not inside a capture
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        warm.step_groups(static)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        g_res = graph_pool.step_groups(static)
    for k in range(4):
        perm = torch.from_numpy(rng.permutation(P).astype(np.int32)).cuda()
        r0 = 0
        eager_groups = []
        for (sx, si), (n, T) in zip(static, SERVER_MIX):
            x = (0.5 * torch.randn(n, 1, T, device="cuda")).clamp_(-1, 1)
            sx.copy_(x)
            si.copy_(perm[r0 : r0 + n])
            eager_groups.append((x, perm[r0 : r0 + n]))
            r0 += n
        graph.replay()
        want = eager.step_groups(eager_groups)
        for (o, y), (o_r, y_r) in zip(g_res, want):
            assert torch.equal(y, y_r) and torch.equal(o, o_r), k
        _assert_pools_equal(graph_pool, eager, k)


class _Group(ctypes.Structure):
    _fields_ = [("ids", ctypes.c_void_p), ("n", ctypes.c_int), ("T", ctypes.c_long), ("x", ctypes.c_void_p), ("y", ctypes.c_void_p),
                ("out", ctypes.c_void_p)]


def _cabi(pq):
    c = pq._lib.cabi
    vp, i, u = ctypes.c_void_p, ctypes.c_int, ctypes.c_uint
    gp = ctypes.POINTER(_Group)
    c.pqmf_stream_pool_analysis_groups_f32.argtypes = [gp, i, vp, vp, vp, vp, i, i, i, u, vp]
    c.pqmf_stream_pool_synthesis_groups_f32.argtypes = [gp, i, vp, vp, vp, vp, i, i, i, u, vp]
    c.pqmf_stream_pool_step_groups_f32.argtypes = [gp, i, vp, vp, vp, vp, vp, vp, i, i, i, u, vp]
    for f in (c.pqmf_stream_pool_analysis_groups_f32, c.pqmf_stream_pool_synthesis_groups_f32, c.pqmf_stream_pool_step_groups_f32):
        f.restype = ctypes.c_int
    return c


@pytest.mark.gpu
def test_group_errors(pq):
    mod = pq.CachedPQMF(100, 16).cuda()
    pool = pq.StreamPool(mod, 64)
    x = torch.zeros(3, 1, 256, device="cuda")
    launches = pq.launch_count()
    with pytest.raises(ValueError, match="across all groups"):
        pool.step_groups([(x, [0, 1, 2]), (x, [3, 4, 0])])
    with pytest.raises(ValueError, match="at most 8"):
        pool.step_groups([(x, [3 * k, 3 * k + 1, 3 * k + 2]) for k in range(9)])
    with pytest.raises(ValueError):
        pool.forward_groups([(x, [0, 1, 1])])
    for dt, name in ((torch.float16, "Half"), (torch.bfloat16, "BFloat16")):
        with pytest.raises(RuntimeError, match=name):
            pool.step_groups([(x, [0, 1, 2]), (x.to(dt), [3, 4, 5])])
        with pytest.raises(RuntimeError, match=name):
            pool.inverse_groups([(torch.zeros(3, 16, 16, device="cuda"), [0, 1, 2]), (torch.zeros(3, 16, 16, device="cuda", dtype=dt), [3, 4, 5])])
    with pytest.raises(RuntimeError, match="not differentiable"):
        pool.step_groups([(x, [0, 1, 2]), (x.clone().requires_grad_(), [3, 4, 5])])
    with pytest.raises(RuntimeError, match="not differentiable"):
        pool.forward_groups([(x.clone().requires_grad_(), [0, 1, 2])])
    with pytest.raises(RuntimeError, match="not differentiable"):
        pool.inverse_groups([(torch.zeros(3, 16, 16, device="cuda", requires_grad=True), [0, 1, 2])])
    with pytest.raises(RuntimeError):  # 3 rows, 2 ids
        pool.step_groups([(x, [0, 1, 2]), (x, torch.tensor([4, 5], device="cuda"))])
    assert pq.launch_count() == launches
    assert (pool.xphase == 0).all() and (pool.sphase == 0).all()
    assert pool.step_groups([]) == [] and pool.step_groups([(x[:0], [])])[0][0].shape == (0, 1, 256)
    assert pq.launch_count() == launches
    # the C entry writes only inside its buffers: guard margins around every group's outputs stay intact
    c = _cabi(pq)
    P, guard = 1200, 1024
    shapes = SERVER_MIX[:2] + ((50, 48),)
    big = StreamPoolGuards(shapes, mod.n_band, guard)
    pool = pq.StreamPool(mod, P)
    ids = torch.randperm(P, device="cuda").to(torch.int32)
    arr, r0 = (_Group * len(shapes))(), 0
    keep = []
    for k, (n, T) in enumerate(shapes):
        x = big.x[k]
        x.copy_(_blocks(n, T, k).reshape(-1))
        gi = ids[r0 : r0 + n].contiguous()
        keep.append(gi)
        arr[k] = _Group(gi.data_ptr(), n, T, x.data_ptr(), big.y[k].data_ptr(), big.out[k].data_ptr())
        r0 += n
    st = torch.cuda.current_stream().cuda_stream
    rc = c.pqmf_stream_pool_step_groups_f32(arr, len(shapes), mod.hk.data_ptr(), mod._tables.data_ptr(), pool.xpool.data_ptr(),
                                            pool.xphase.data_ptr(), pool.spool.data_ptr(), pool.sphase.data_ptr(), P, mod.n_band,
                                            mod.hk.shape[1], mod._flags, st)
    assert rc == 0
    torch.cuda.synchronize()
    big.check()


class StreamPoolGuards:
    """x, y and out of every group inside buffers with `guard` sentinel floats on both sides."""

    SENTINEL = 12345.0

    def __init__(self, shapes, m, guard):
        self.guard, self.bufs = guard, []
        self.x, self.y, self.out = [], [], []
        for n, T in shapes:
            for lst in (self.x, self.y, self.out):
                buf = torch.full((n * T + 2 * guard,), self.SENTINEL, device="cuda")
                self.bufs.append(buf)
                lst.append(buf[guard : guard + n * T])

    def check(self):
        for buf in self.bufs:
            assert (buf[: self.guard] == self.SENTINEL).all() and (buf[-self.guard :] == self.SENTINEL).all()


def test_group_cabi_argument_checks_happen_before_any_cuda_call(pq):
    """The grouped entries validate on the host and return PQMF_ERR_ARG (or 0 when there are no rows) without touching a device."""
    c = _cabi(pq)
    an, sy, st = c.pqmf_stream_pool_analysis_groups_f32, c.pqmf_stream_pool_synthesis_groups_f32, c.pqmf_stream_pool_step_groups_f32
    fake = 4096  # never dereferenced: every call below fails a host check or has no rows

    def groups(*specs):
        arr = (_Group * max(len(specs), 1))()
        for k, (n, T, ptrs) in enumerate(specs):
            arr[k] = _Group(fake if ptrs else None, n, T, fake if ptrs else None, fake if ptrs else None, fake if ptrs else None)
        return arr

    def call(f, arr, G, P=64, M=16, L=512, pools=True):
        p = fake if pools else None
        if f is st:
            return f(arr, G, fake, None, p, p, p + 8 if pools else None, p + 8 if pools else None, P, M, L, 0, None)
        return f(arr, G, fake, None, p, p, P, M, L, 0, None)

    for f in (an, sy, st):
        assert call(f, groups(), 0) == 0                                  # G == 0
        assert call(f, groups((0, 512, False), (0, 2048, False)), 2) == 0  # all empty
        assert call(f, groups((0, 512, False)), 1, pools=False) == 0     # all empty, no pools
        assert call(f, groups(), -1) == -1                                # G < 0
        assert call(f, groups(*[(1, 512, True)] * 9), 9) == -1            # G > 8
        assert call(f, None, 2) == -1                                     # no descriptors
        assert call(f, groups((40, 512, True), (30, 512, True)), 2) == -1  # more rows than P
        assert call(f, groups((4, 520, True), (4, 512, True)), 2) == -1   # T % M != 0
        assert call(f, groups((4, 0, True), (4, 512, True)), 2) == -1     # T == 0
        assert call(f, groups((4, 512, False), (4, 512, True)), 2) == -1  # null pointers in a non-empty group
        assert call(f, groups((-1, 512, True)), 1) == -1                  # n < 0
        assert call(f, groups((4, 512, True)), 1, P=0) == -1              # P < 1
        assert call(f, groups((4, 512, True), (4, 512, True)), 2, pools=False) == -1  # null pool
    # a step needs two distinct phase arrays
    arr = groups((4, 512, True), (4, 512, True))
    assert st(arr, 2, fake, None, fake, fake, fake, fake, 64, 16, 512, 0, None) == -1
