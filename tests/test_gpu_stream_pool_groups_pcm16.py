"""Grouped stream-pool calls with 16-bit PCM blocks: StreamPool.step_groups_pcm16 / forward_groups_pcm16 / inverse_groups_pcm16 and
pqmf_stream_pool_*_groups_pcm16.

Every call must give, per row, the bits of the fp32 grouped call (step_groups / forward_groups / inverse_groups) on the widened blocks,
followed by quantising, with the same pool and phase-word updates -- so each test drives a twin pool with the fp32 grouped calls and
compares outputs, both state halves and the phase words.  The joined groups are the fp32 call's; a joined group that cannot run natively
(misaligned PCM, interleaved stereo output) makes the C entry refuse the whole call with nothing launched, and a group the grouped launch
does not take whose single-group PCM entry refuses is marked in the `staged` mask.  The last test needs no GPU: it checks the C entries'
argument validation."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import pqmf_oracle as O

TOL = 1e-5
MIN_TILES = 96
ERR_ARG, ERR_UNSUPPORTED = -1, -2
FLAG_BLOCKERS = 2 | 4 | 8 | 16 | (1 << 23)  # NO_SIGN, FOLD, NO_PAIR, FP32, H4_SPLIT


@pytest.fixture(scope="module")
def pq():
    import pqmf_b200

    return pqmf_b200


def widen(pcm, downmix):
    """[S, T, C] int16 -> [S, C', T] float32, the kernels' arithmetic (the down-mix summed in channel order, then / C)."""
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


def pcm_blocks(S, T, C, seed, scale=8000.0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (scale * torch.randn(S, T, C, device="cuda", generator=g)).round().clamp(-32768, 32767).to(torch.int16)


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


def _joined(mod, shapes):
    """Indices of the groups (rows, T) that run in the grouped launch of a step (the fp32 rule: aligned fresh blocks)."""
    if len(shapes) < 2:
        return set()
    plan = {k: _spt(mod, T) for k, (n, T) in enumerate(shapes) if n > 0 and _spt(mod, T) is not None}
    ta = sum(_tiles(shapes[k][0], s[0]) for k, s in plan.items())
    ts = sum(_tiles(shapes[k][0], s[1]) for k, s in plan.items())
    return set(plan) if len(plan) >= 2 and ta >= MIN_TILES and ts >= MIN_TILES else set()


def _state(pool):
    return [t.clone() for t in (pool.xpool, pool.spool, pool.xphase, pool.sphase)]


def _assert_pools_equal(a, b, what=""):
    for u, v in zip((a.xpool, a.spool, a.xphase, a.sphase), (b.xpool, b.spool, b.xphase, b.sphase)):
        assert torch.equal(u, v), what


def _split(P, sizes, seed=0):
    perm = torch.randperm(P, generator=torch.Generator().manual_seed(seed)).to(torch.int32).cuda()
    ids, r0 = [], 0
    for n in sizes:
        ids.append(perm[r0 : r0 + n])
        r0 += n
    return ids


def twin_step(twin, groups, downmix):
    """step_groups_pcm16 as the fp32 grouped step on the widened blocks, then quantised."""
    xs = [(widen(p, downmix).reshape(-1, 1, p.shape[1]), i) for p, i in groups]
    res = []
    for (p, _), (o, y) in zip(groups, twin.step_groups(xs)):
        S, T = p.shape[0], p.shape[1]
        res.append((quantise(o.view(S, -1, T)), y.view(S, -1, y.shape[-1])))
    return res


def twin_forward(twin, groups, downmix):
    xs = [(widen(p, downmix).reshape(-1, 1, p.shape[1]), i) for p, i in groups]
    return [y.view(p.shape[0], -1, y.shape[-1]) for (p, _), y in zip(groups, twin.forward_groups(xs))]


def twin_inverse(twin, groups, m):
    ss = [(s.reshape(-1, m, s.shape[-1]), i) for s, i in groups]
    return [quantise(o.view(s.shape[0], -1, o.shape[-1])) for (s, _), o in zip(groups, twin.inverse_groups(ss))]


def _assert_results_equal(got, want, what=""):
    for k, (g, w) in enumerate(zip(got, want)):
        if isinstance(g, tuple):
            assert torch.equal(g[0], w[0]) and torch.equal(g[1], w[1]), (what, k)
        else:
            assert torch.equal(g, w), (what, k)


# ---- the C entries ----
class _Group(ctypes.Structure):
    _fields_ = [("ids", ctypes.c_void_p), ("n", ctypes.c_int), ("T", ctypes.c_long), ("C", ctypes.c_int), ("pcm", ctypes.c_void_p),
                ("y", ctypes.c_void_p), ("pcm_out", ctypes.c_void_p)]


def _cabi(pq):
    c = pq._lib.cabi
    vp, i, u = ctypes.c_void_p, ctypes.c_int, ctypes.c_uint
    gp, up = ctypes.POINTER(_Group), ctypes.POINTER(ctypes.c_uint)
    c.pqmf_stream_pool_analysis_groups_pcm16.argtypes = [gp, i, i, vp, vp, vp, vp, i, i, i, u, up, vp]
    c.pqmf_stream_pool_synthesis_groups_pcm16.argtypes = [gp, i, vp, vp, vp, vp, i, i, i, u, up, vp]
    c.pqmf_stream_pool_step_groups_pcm16.argtypes = [gp, i, i, vp, vp, vp, vp, vp, vp, i, i, i, u, up, vp]
    for f in (c.pqmf_stream_pool_analysis_groups_pcm16, c.pqmf_stream_pool_synthesis_groups_pcm16, c.pqmf_stream_pool_step_groups_pcm16):
        f.restype = ctypes.c_int
    return c


def c_step(pq, mod, pool, groups, downmix, outs=None):
    """pqmf_stream_pool_step_groups_pcm16 on (pcm, ids) groups: (rc, staged, launches, [(pcm_out, y)])."""
    c = _cabi(pq)
    m = mod.n_band
    arr = (_Group * max(len(groups), 1))()
    res = []
    for k, (p, i) in enumerate(groups):
        S, T, C = p.shape
        Cr = 1 if downmix else C
        o, y = outs[k] if outs else (torch.empty(S, T, Cr, dtype=torch.int16, device="cuda"), torch.empty(S, Cr * m, T // m, device="cuda"))
        res.append((o, y))
        arr[k] = _Group(i.data_ptr(), S, T, C, p.data_ptr(), y.data_ptr(), o.data_ptr())
    staged = ctypes.c_uint(0xFFFF)
    launches = pq.launch_count()
    rc = c.pqmf_stream_pool_step_groups_pcm16(arr, len(groups), int(downmix), mod.hk.data_ptr(), mod._tables.data_ptr(), pool.xpool.data_ptr(),
                                               pool.xphase.data_ptr(), pool.spool.data_ptr(), pool.sphase.data_ptr(), pool.capacity, m,
                                               mod.hk.shape[1], mod._flags, ctypes.byref(staged), torch.cuda.current_stream().cuda_stream)
    return rc, staged.value, pq.launch_count() - launches, res


# n_band -> block lengths whose groups each run the streaming Hankel-4 kernels (7680 at n_band 16: the largest native block)
NATIVE = {8: (512, 1024, 2048), 16: (512, 2048, 7680), 32: (1024, 2048, 4096)}


@pytest.mark.gpu
@pytest.mark.parametrize("m", (8, 16, 32))
@pytest.mark.parametrize("C,downmix", ((1, False), (2, True), (2, False)))
def test_native_groups_equal_the_fp32_twin(pq, m, C, downmix):
    """Mono and stereo groups at every native block length.  A step makes 3 launches, forward or inverse 2; stereo rows without down-mix
    run natively in the analysis and are refused (nothing launched) by the step, whose output would be interleaved."""
    mod = pq.CachedPQMF(100, m).cuda()
    Cr = 1 if downmix else C
    shapes = []  # (clips, T)
    for T in NATIVE[m]:
        s = _spt(mod, T)
        assert s is not None, (m, T)
        shapes.append((-(-(MIN_TILES * max(s) + 5) // Cr), T))
    P = sum(n * Cr for n, _ in shapes) + 64
    a, b = pq.StreamPool(mod, P), pq.StreamPool(mod, P)
    ids = _split(P, [n * Cr for n, _ in shapes], m)
    for step in range(2):
        groups = [(pcm_blocks(n, T, C, 100 * step + k), ids[k]) for k, (n, T) in enumerate(shapes)]
        want = twin_step(b, groups, downmix)
        if Cr == 1:
            rc, staged, launches, got = c_step(pq, mod, a, groups, downmix)
            assert (rc, staged, launches) == (0, 0, 3), step
        else:
            before = _state(a)
            rc, staged, launches, _ = c_step(pq, mod, a, groups, downmix)
            assert (rc, launches) == (ERR_UNSUPPORTED, 0), step
            for u, v in zip(_state(a), before):
                assert torch.equal(u, v)
            got = a.step_groups_pcm16(groups, downmix=downmix)
        _assert_results_equal(got, want, step)
        _assert_pools_equal(a, b, step)
    groups = [(pcm_blocks(n, T, C, 7 + k), ids[k]) for k, (n, T) in enumerate(shapes)]
    launches = pq.launch_count()
    ys = a.forward_groups_pcm16(groups, downmix=downmix)
    assert pq.launch_count() - launches == 2
    _assert_results_equal(ys, twin_forward(b, groups, downmix))
    _assert_pools_equal(a, b)
    if Cr == 1:
        launches = pq.launch_count()
        outs = a.inverse_groups_pcm16([(y, i) for y, (_, i) in zip(ys, groups)])
        assert pq.launch_count() - launches == 2
        _assert_results_equal(outs, twin_inverse(b, [(y, i) for y, (_, i) in zip(ys, groups)], m))
        _assert_pools_equal(a, b)


SERVER_MIX = ((600, 512), (400, 1024), (250, 2048), (90, 4096))  # n_band 16: 75 + 80 + 84 + 90 tiles, each below 96 alone


@pytest.mark.gpu
def test_server_mix_reaches_the_tensor_cores_together(pq):
    mod = pq.CachedPQMF(100, 16).cuda()
    assert _joined(mod, SERVER_MIX) == {0, 1, 2, 3}
    P = 2048
    pool, twin, alone = pq.StreamPool(mod, P), pq.StreamPool(mod, P), pq.StreamPool(mod, P)
    ids = _split(P, [n for n, _ in SERVER_MIX], 1)
    for step in range(2):
        groups = [(pcm_blocks(n, T, 1, 10 * step + k), ids[k]) for k, (n, T) in enumerate(SERVER_MIX)]
        launches = pq.launch_count()
        got = pool.step_groups_pcm16(groups)
        assert pq.launch_count() - launches == 3
        want = twin_step(twin, groups, False)
        direct = [alone.step_pcm16(p, i) for p, i in groups]  # each group alone is below the threshold: staged onto the direct form
        _assert_results_equal(got, want, step)
        for k, ((o, y), (o_d, y_d)) in enumerate(zip(got, direct)):
            assert not torch.equal(y, y_d), (step, k)
        _assert_pools_equal(pool, twin, step)


def _check_oracle(mod, before, pcm, y, out, ids, rows, what):
    """Rows of one mono group against the float64 oracle on the widened input: sub-bands within TOL / 2, PCM output within one LSB of the
    quantised oracle."""
    m, length = mod.hk.shape
    hk = mod.hk.cpu().double().numpy()
    xpool, spool, xphase, sphase = before
    x = widen(pcm, False)
    for r in rows:
        i = int(ids[r])
        st = O.StreamState(1, m, length)
        st.x_hist = xpool[int(xphase[i]) & 1, i].cpu().double().numpy()[None]
        st.s_hist = spool[int(sphase[i]) & 1, i].cpu().double().numpy()[None]
        st.frames_in, st.frames_out = (int(xphase[i]) >> 1) & 1, (int(sphase[i]) >> 1) & 1
        y64 = O.stream_analysis(x[r : r + 1, 0].cpu().double().numpy(), hk, st)
        o64 = O.stream_synthesis(y[r : r + 1].cpu().double().numpy(), hk, st)
        assert np.abs(y[r : r + 1].cpu().numpy() - y64).max() <= TOL / 2, (what, r)
        q64 = np.clip(np.rint(o64 * 32768.0), -32768, 32767)
        assert np.abs(out[r, :, 0].cpu().numpy().astype(np.int64) - q64[0]).max() <= 1, (what, r)


@pytest.mark.gpu
def test_steady_state_across_group_boundaries(pq):
    """About ten tiles per CTA over four groups, an odd tile count and a one-stream last tile in each group; oracle rows on every CTA's
    first three and last tiles and on both sides of every group boundary (a PCM analysis that widened a tile with the previous group's
    frames would fail there)."""
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
    ids = _split(P, [n for n, _ in shapes], 2)
    tile0 = np.cumsum([0] + tiles)
    picks = set()
    for c in range(grid):
        its = list(range(c, total, grid))
        picks.update(its[:3] + its[-1:])
    for k in range(1, 4):
        picks.update((tile0[k] - 1, tile0[k]))
    for step in range(2):
        groups = [(pcm_blocks(n, T, 1, 50 + 10 * step + k), ids[k]) for k, (n, T) in enumerate(shapes)]
        before = _state(a)
        launches = pq.launch_count()
        got = a.step_groups_pcm16(groups)
        assert pq.launch_count() - launches == 3
        _assert_results_equal(got, twin_step(b, groups, False), step)
        _assert_pools_equal(a, b, step)
        if step == 1:
            for t in sorted(picks):
                k = int(np.searchsorted(tile0, t, side="right") - 1)
                spt = _spt(mod, shapes[k][1])[0]
                row = (t - tile0[k]) * spt
                last = min(row + spt, shapes[k][0]) - 1
                p, i = groups[k]
                o, y = got[k]
                _check_oracle(mod, before, p, y, o, i, sorted({row, last}), (t, k))


@pytest.mark.gpu
def test_refused_groups(pq):
    """480- and 48-sample groups next to joined ones are marked in `staged` (their single-group PCM entry refuses) while the rest runs
    natively; a misaligned PCM view or stereo output in a joined group refuses the whole call with nothing launched.  Through the op every
    case equals the twin."""
    mod = pq.CachedPQMF(100, 16).cuda()
    P = 3072
    pool, twin = pq.StreamPool(mod, P), pq.StreamPool(mod, P)
    shapes = [(600, 512), (200, 480), (400, 1024), (50, 48), (300, 2048)]
    assert _joined(mod, shapes) == {0, 2, 4}
    ids = _split(P, [n for n, _ in shapes], 3)
    for step in range(2):
        groups = [(pcm_blocks(n, T, 1, 30 + 10 * step + k), i) for k, ((n, T), i) in enumerate(zip(shapes, ids))]
        want = twin_step(twin, groups, False)
        rc, staged, launches, got = c_step(pq, mod, pool, groups, False)
        assert (rc, staged, launches) == (0, 0b01010, 3), step
        for k in (1, 3):  # what the op does for a staged group
            got[k] = pool.step_pcm16(*groups[k])
        _assert_results_equal(got, want, step)
        _assert_pools_equal(pool, twin, step)
        # the same through the op
        got = pool.step_groups_pcm16(groups)
        _assert_results_equal(got, twin_step(twin, groups, False), step)
        _assert_pools_equal(pool, twin, step)
    # a misaligned PCM view (2 bytes into its storage) in a joined group
    groups = [(pcm_blocks(n, T, 1, 90 + k), i) for k, ((n, T), i) in enumerate(zip(shapes, ids))]
    n, T = shapes[2]
    buf = torch.empty(n * T + 1, dtype=torch.int16, device="cuda")
    buf[1:].copy_(groups[2][0].reshape(-1))
    groups[2] = (buf[1:].view(n, T, 1), ids[2])
    assert groups[2][0].is_contiguous() and groups[2][0].data_ptr() % 32 != 0
    before = _state(pool)
    rc, _, launches, _ = c_step(pq, mod, pool, groups, False)
    assert (rc, launches) == (ERR_UNSUPPORTED, 0)
    for u, v in zip(_state(pool), before):
        assert torch.equal(u, v)
    _assert_results_equal(pool.step_groups_pcm16(groups), twin_step(twin, groups, False))
    _assert_pools_equal(pool, twin)
    # stereo output without down-mix in a joined group: the joined set is the fp32 call's on the stereo group's rows
    sizes = [600, 200, 200, 50, 300]
    groups = [(pcm_blocks(sizes[k] // (2 if k == 2 else 1), T, 2 if k == 2 else 1, 95 + k), ids[k][: sizes[k]])
              for k, (_, T) in enumerate(shapes)]
    rc, _, launches, _ = c_step(pq, mod, pool, groups, False)
    assert (rc, launches) == (ERR_UNSUPPORTED, 0)
    _assert_results_equal(pool.step_groups_pcm16(groups), twin_step(twin, groups, False))
    _assert_pools_equal(pool, twin)


@pytest.mark.gpu
def test_saturation_and_ties(pq):
    """Blocks loud enough to saturate the output at both ends; the twin's outputs include exact .5 ties of v * 32768, which both sides
    round to even."""
    mod = pq.CachedPQMF(100, 16).cuda()
    shapes = SERVER_MIX
    P = 2048
    pool, twin = pq.StreamPool(mod, P), pq.StreamPool(mod, P)
    ids = _split(P, [n for n, _ in shapes], 4)
    saw_max = saw_min = 0
    ties = 0
    for step in range(3):
        groups = []
        for k, (n, T) in enumerate(shapes):
            g = torch.Generator(device="cuda").manual_seed(200 + 10 * step + k)
            sq = torch.where(torch.rand(n, T // 64, 1, device="cuda", generator=g) < 0.5, -32768, 32767).repeat_interleave(64, 1)
            groups.append((sq.to(torch.int16), ids[k]))
        got = pool.step_groups_pcm16(groups)
        xs = [(widen(p, False).reshape(-1, 1, p.shape[1]), i) for p, i in groups]
        fp = twin.step_groups(xs)
        for (o, y), (of, yf), (p, _) in zip(got, fp, groups):
            assert torch.equal(y, yf.view_as(y)) and torch.equal(o, quantise(of)), step
            v = of * 32768.0
            ties += int(((v - v.floor()) == 0.5).sum())
            saw_max += int((o == 32767).sum())
            saw_min += int((o == -32768).sum())
        _assert_pools_equal(pool, twin, step)
    assert saw_max > 0 and saw_min > 0 and ties > 0, (saw_max, saw_min, ties)


@pytest.mark.gpu
def test_seeded_schedule_over_a_pool(pq):
    """Twelve steps over a pool of 4096 mixing step_groups_pcm16, step_groups, step_pcm16 and step on the same streams, with resets and a dead
    CUDA id; against the twin driven by the fp32 calls on the widened blocks.  Streams not listed keep both halves and their phase words."""
    P = 4096
    mod = pq.CachedPQMF(100, 16).cuda()
    pool, twin = pq.StreamPool(mod, P), pq.StreamPool(mod, P)
    rng = np.random.default_rng(11)
    lengths = (48, 256, 480, 512, 1024, 2048, 4096)
    for step in range(12):
        if step in (4, 9):
            gone = rng.choice(P, 500, replace=False).tolist()
            pool.reset(gone)
            twin.reset(gone)
        kind = ("groups_pcm16", "groups_pcm16", "groups", "pcm16", "groups_pcm16", "plain")[step % 6]
        G = int(rng.integers(2, 9)) if kind.startswith("groups") else 1
        n_all = int(rng.integers(G, 3000))
        chosen = rng.choice(P, n_all, replace=False)
        parts = np.split(chosen, np.sort(rng.choice(np.arange(1, n_all), G - 1, replace=False))) if G > 1 else [chosen]
        groups = []
        for k, part in enumerate(parts):
            T = int(rng.choice(lengths))
            groups.append((pcm_blocks(len(part), T, 1, 1000 * step + k), torch.from_numpy(part.astype(np.int32)).cuda()))
        dead = step == 6
        if dead:  # one dead row in the first group: an id outside [0, P)
            p0, i0 = groups[0]
            groups[0] = (torch.cat([p0, pcm_blocks(1, p0.shape[1], 1, 5)]), torch.cat([i0, torch.tensor([P + 3], dtype=torch.int32, device="cuda")]))
        before = _state(pool)
        live = [(p[:-1], i[:-1]) if dead and k == 0 else (p, i) for k, (p, i) in enumerate(groups)]
        if kind == "groups_pcm16":
            got = pool.step_groups_pcm16(groups)
            want = twin_step(twin, groups, False)  # the dead row too: the same rows, so the same joined set
        elif kind == "groups":
            got = pool.step_groups([(widen(p, False), i) for p, i in groups])
            want = twin.step_groups([(widen(p, False), i) for p, i in groups])
        elif kind == "pcm16":
            got = [pool.step_pcm16(*groups[0])]
            o, y = twin.step(widen(groups[0][0], False), groups[0][1])
            want = [(quantise(o), y)]
        else:
            got = [pool.step(widen(groups[0][0], False), groups[0][1])]
            want = [twin.step(widen(groups[0][0], False), groups[0][1])]
        for k, ((o, y), (o_r, y_r)) in enumerate(zip(got, want)):
            assert torch.equal(y, y_r) and torch.equal(o, o_r), (step, kind, k)
            if dead and k == 0:
                assert (y[-1] == 0).all() and (o[-1] == 0).all()
        _assert_pools_equal(pool, twin, step)
        listed = torch.cat([i for _, i in live]).long()
        rest = torch.ones(P, dtype=torch.bool, device="cuda")
        rest[listed] = False
        for now, then in zip(_state(pool), before):
            assert torch.equal(now[:, rest] if now.dim() > 1 else now[rest], then[:, rest] if then.dim() > 1 else then[rest]), step


@pytest.mark.gpu
def test_one_graph_replays_grouped_pcm_steps(pq):
    mod = pq.CachedPQMF(100, 16).cuda()
    P = 2048
    graph_pool, eager = pq.StreamPool(mod, P), pq.StreamPool(mod, P)
    rng = np.random.default_rng(3)
    pre = torch.from_numpy(rng.choice(P, P // 3, replace=False).astype(np.int32)).cuda()  # mixed parities, identically on both pools
    xpre = pcm_blocks(pre.numel(), 48, 1, 1)
    graph_pool.step_pcm16(xpre, pre)
    eager.step_pcm16(xpre, pre)
    static = [(torch.zeros(n, T, 1, dtype=torch.int16, device="cuda"), torch.arange(r0, r0 + n, dtype=torch.int32, device="cuda"))
              for (n, T), r0 in zip(SERVER_MIX, np.cumsum([0] + [n for n, _ in SERVER_MIX])[:-1].tolist())]
    warm = pq.StreamPool(mod, P)  # first launches set the kernels' shared-memory limits: not inside a capture
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        warm.step_groups_pcm16(static)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        g_res = graph_pool.step_groups_pcm16(static)
    for k in range(4):
        perm = torch.from_numpy(rng.permutation(P).astype(np.int32)).cuda()
        r0 = 0
        eager_groups = []
        for (sp, si), (n, T) in zip(static, SERVER_MIX):
            p = pcm_blocks(n, T, 1, 300 + 10 * k + r0 % 7)
            sp.copy_(p)
            si.copy_(perm[r0 : r0 + n])
            eager_groups.append((p, perm[r0 : r0 + n]))
            r0 += n
        graph.replay()
        _assert_results_equal(g_res, eager.step_groups_pcm16(eager_groups), k)
        _assert_pools_equal(graph_pool, eager, k)


@pytest.mark.gpu
def test_group_pcm_errors_and_buffer_bounds(pq):
    mod = pq.CachedPQMF(100, 16).cuda()
    pool = pq.StreamPool(mod, 64)
    p = torch.zeros(3, 256, 1, dtype=torch.int16, device="cuda")
    s = torch.zeros(3, 16, 16, device="cuda")
    launches = pq.launch_count()
    with pytest.raises(ValueError, match="across all groups"):
        pool.step_groups_pcm16([(p, [0, 1, 2]), (p, [3, 4, 0])])
    with pytest.raises(ValueError, match="at most 8"):
        pool.forward_groups_pcm16([(p, [3 * k, 3 * k + 1, 3 * k + 2]) for k in range(9)])
    with pytest.raises(ValueError):
        pool.inverse_groups_pcm16([(s, [0, 1, 1])])
    with pytest.raises(RuntimeError, match="int16"):
        pool.step_groups_pcm16([(p, [0, 1, 2]), (p.float(), [3, 4, 5])])
    with pytest.raises(RuntimeError, match="int16"):
        pool.forward_groups_pcm16([(p.to(torch.int32), [0, 1, 2])])
    with pytest.raises(RuntimeError):  # 2 channels without down-mix: 6 rows, 3 ids
        pool.step_groups_pcm16([(torch.zeros(3, 256, 2, dtype=torch.int16, device="cuda"), [0, 1, 2])])
    with pytest.raises(RuntimeError, match="multiple of n_band"):
        pool.step_groups_pcm16([(torch.zeros(3, 250, 1, dtype=torch.int16, device="cuda"), [0, 1, 2])])
    with pytest.raises(RuntimeError, match="Half"):
        pool.inverse_groups_pcm16([(s, [0, 1, 2]), (s.half(), [3, 4, 5])])
    with pytest.raises(RuntimeError, match="not differentiable"):
        pool.inverse_groups_pcm16([(s.clone().requires_grad_(), [0, 1, 2])])
    with pytest.raises(RuntimeError, match="more rows"):
        pool.step_groups_pcm16([(torch.zeros(40, 256, 1, dtype=torch.int16, device="cuda"), torch.arange(40, dtype=torch.int32, device="cuda")),
                                (torch.zeros(30, 256, 1, dtype=torch.int16, device="cuda"), torch.arange(30, dtype=torch.int32, device="cuda"))])
    assert pq.launch_count() == launches
    assert (pool.xphase == 0).all() and (pool.sphase == 0).all()
    assert pool.step_groups_pcm16([]) == [] and pool.step_groups_pcm16([(p[:0], [])])[0][0].shape == (0, 256, 1)
    assert pool.forward_groups_pcm16([(p[:0], [])])[0].shape == (0, 16, 16)
    assert pool.inverse_groups_pcm16([(s[:0], [])])[0].shape == (0, 256, 1)
    assert pq.launch_count() == launches
    # the C entry writes only inside its buffers: guard margins around every group's pcm_out and y, joined and staged groups
    P, guard = 1300, 1024
    shapes = SERVER_MIX[:2] + ((50, 48), (60, 480))
    pool = pq.StreamPool(mod, P)
    ids = _split(P, [n for n, _ in shapes], 5)
    bufs, outs, groups = [], [], []
    for k, (n, T) in enumerate(shapes):
        ob = torch.full((n * T + 2 * guard,), 12345, dtype=torch.int16, device="cuda")
        yb = torch.full((n * T + 2 * guard,), 12345.0, device="cuda")
        bufs += [ob, yb]
        outs.append((ob[guard : guard + n * T].view(n, T, 1), yb[guard : guard + n * T].view(n, 16, T // 16)))
        groups.append((pcm_blocks(n, T, 1, k), ids[k]))
    rc, staged, launches, _ = c_step(pq, mod, pool, groups, False, outs)
    assert (rc, staged, launches) == (0, 0b1100, 3)
    torch.cuda.synchronize()
    for b in bufs:
        assert (b[:guard] == 12345).all() and (b[-guard:] == 12345).all()


def test_group_pcm_cabi_argument_checks_happen_before_any_cuda_call(pq):
    """The grouped PCM entries validate on the host and return PQMF_ERR_ARG (or 0 when there are no rows) without touching a device."""
    c = _cabi(pq)
    an, sy, st = c.pqmf_stream_pool_analysis_groups_pcm16, c.pqmf_stream_pool_synthesis_groups_pcm16, c.pqmf_stream_pool_step_groups_pcm16
    fake = 4096  # never dereferenced: every call below fails a host check or has no rows

    def groups(*specs):
        arr = (_Group * max(len(specs), 1))()
        for k, (n, T, C, ptrs) in enumerate(specs):
            q = fake if ptrs else None
            arr[k] = _Group(q, n, T, C, q, q, q)
        return arr

    def call(f, arr, G, P=64, M=16, L=512, pools=True, staged=True, downmix=0):
        p = fake if pools else None
        mask = ctypes.c_uint(77)
        sp = ctypes.byref(mask) if staged else None
        if f is st:
            return f(arr, G, downmix, fake, None, p, p, p + 8 if pools else None, p + 8 if pools else None, P, M, L, 0, sp, None)
        if f is an:
            return f(arr, G, downmix, fake, None, p, p, P, M, L, 0, sp, None)
        return f(arr, G, fake, None, p, p, P, M, L, 0, sp, None)

    for f in (an, sy, st):
        assert call(f, groups(), 0) == 0                                          # G == 0
        assert call(f, groups((0, 512, 1, False), (0, 2048, 2, False)), 2) == 0     # all empty
        assert call(f, groups((0, 512, 1, False)), 1, pools=False) == 0          # all empty, no pools
        assert call(f, groups(), -1) == -1                                        # G < 0
        assert call(f, groups(*[(1, 512, 1, True)] * 9), 9) == -1                 # G > 8
        assert call(f, None, 2) == -1                                             # no descriptors
        assert call(f, groups((40, 512, 1, True), (30, 512, 1, True)), 2) == -1   # more rows than P
        assert call(f, groups((20, 512, 2, True), (30, 512, 1, True)), 2) == -1   # more rows than P: 2 channels
        assert call(f, groups((4, 520, 1, True), (4, 512, 1, True)), 2) == -1     # T % M != 0
        assert call(f, groups((4, 0, 1, True), (4, 512, 1, True)), 2) == -1       # T == 0
        assert call(f, groups((4, 512, 0, True), (4, 512, 1, True)), 2) == -1     # C < 1
        assert call(f, groups((4, 512, 65, True)), 1, P=4096) == -1               # C > 64
        assert call(f, groups((0, 512, 0, False)), 1) == -1                       # C < 1 in an empty group
        assert call(f, groups((4, 512, 1, False), (4, 512, 1, True)), 2) == -1    # null pointers in a non-empty group
        assert call(f, groups((-1, 512, 1, True)), 1) == -1                       # n < 0
        assert call(f, groups((4, 512, 1, True)), 1, P=0) == -1                   # P < 1
        assert call(f, groups((4, 512, 1, True), (4, 512, 1, True)), 2, pools=False) == -1  # null pool
        assert call(f, groups((4, 512, 1, True)), 1, staged=False) == -1          # null staged
        assert call(f, groups(), 0, staged=False) == -1                           # null staged, no groups
    # a step needs two distinct phase arrays
    arr = groups((4, 512, 1, True), (4, 512, 1, True))
    mask = ctypes.c_uint(0)
    assert st(arr, 2, 0, fake, None, fake, fake, fake, fake, 64, 16, 512, 0, ctypes.byref(mask), None) == -1
