"""Grouped stream-pool calls with bf16 / fp16 blocks: StreamPool(mod, P, dtype).forward_groups / inverse_groups / step_groups and
pqmf_stream_pool_{analysis,synthesis}_groups_x.

Every call must give, per row, the bits of a twin float32 pool driven by forward_groups / inverse_groups on the widened blocks, rounded to
the dtype; step_groups is forward_groups followed by inverse_groups of the ROUNDED sub-bands.  Pool halves and phase words must equal the
twin's.  Each direction joins exactly the groups the float32 call of that direction would join; a joined group whose half buffers are not
16-byte aligned makes the C entry refuse the whole call with nothing launched, and a group the grouped launch does not take whose
single-group half entry refuses is marked in the `staged` mask.  Outputs are compared as bits.  The last test needs no GPU: it checks the C
entries' argument validation."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import pqmf_oracle as O

ERR_ARG, ERR_UNSUPPORTED = -1, -2
DT_F32, DT_F16, DT_BF16 = 0, 1, 2
DTYPES = [torch.float16, torch.bfloat16]
CODE = {torch.float16: DT_F16, torch.bfloat16: DT_BF16}
TOL = 1e-5
MIN_TILES = 96
GUARD = 0x7DAD  # guard half word: a NaN in bf16 and fp16 that no kernel writes
FLAG_BLOCKERS = 2 | 4 | 8 | 16 | (1 << 23)  # NO_SIGN, FOLD, NO_PAIR, FP32, H4_SPLIT


@pytest.fixture(scope="module")
def pq():
    import pqmf_b200

    return pqmf_b200


@pytest.fixture(scope="module")
def mods(pq):
    cache = {}

    def get(att, m):
        if (att, m) not in cache:
            cache[(att, m)] = pq.CachedPQMF(att, m).cuda()
        return cache[(att, m)]

    return get


# ---------------------------------------------------------------- the float32 streaming plan per direction (h4_*_stream_plan), host arithmetic
def _geom(rows_b, hist):
    pitch = (rows_b + hist // 64 + 3) & ~3
    return pitch, 128 // pitch


def _spt(mod, T):
    """(analysis, synthesis) streams per tile of a T-sample block, None in a direction whose streaming Hankel-4 kernels cannot plan it."""
    m, length = mod.hk.shape
    flags = mod._flags
    jlo, kt = 32 * ((flags >> 8) & 0xF), 32 * ((flags >> 12) & 0x1F)
    if m not in (8, 16, 32) or mod._tables.numel() == 0 or kt == 0 or flags & FLAG_BLOCKERS:
        return None, None
    sa = ss = None
    hist_a = -(-(length - jlo) // 64) * 64
    if not (hist_a > length or T % 256 or T < length or length % 8):
        pitch, spt = _geom(T // 64, hist_a)
        sa = spt if pitch <= 128 and spt >= 1 else None
    taps = (jlo + kt) // m
    hist_fr = -(-(taps * m) // 64) * 64 // m
    F, K = T // m, length // m
    if not (hist_fr % 4 or hist_fr > K or (F * m) % 256 or F % 4 or F < K):
        pitch, spt = _geom(T // 64, hist_fr * m)
        ss = spt if pitch <= 128 and spt >= 1 else None
    return sa, ss


def _tiles(n, spt):
    return -(-n // spt)


def _joined(mod, shapes, d):
    """Indices of the groups (rows, T) the float32 grouped call of direction d (0 analysis, 1 synthesis) runs in its grouped launch."""
    plan = {k: _spt(mod, T)[d] for k, (n, T) in enumerate(shapes) if n > 0 and _spt(mod, T)[d] is not None}
    tiles = sum(_tiles(shapes[k][0], s) for k, s in plan.items())
    return set(plan) if len(plan) >= 2 and tiles >= MIN_TILES else set()


# ---------------------------------------------------------------- helpers
def blocks(shape, seed, dtype, scale=0.5):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (scale * torch.randn(shape, device="cuda", generator=g)).clamp_(-1, 1).to(dtype)


def bits_equal(a, b):
    return a.dtype == b.dtype and a.shape == b.shape and torch.equal(a.view(torch.int16), b.view(torch.int16))


def _state(pool):
    return [t.clone() for t in (pool.xpool, pool.spool, pool.xphase, pool.sphase)]


def pools_equal(a, b):
    return all(torch.equal(u, v) for u, v in zip((a.xpool, a.spool, a.xphase, a.sphase), (b.xpool, b.spool, b.xphase, b.sphase)))


def _split(P, sizes, seed=0):
    perm = torch.randperm(P, generator=torch.Generator().manual_seed(seed)).to(torch.int32).cuda()
    ids, r0 = [], 0
    for n in sizes:
        ids.append(perm[r0 : r0 + n])
        r0 += n
    return ids


def twin_forward(twin, groups, dtype):
    return [y.to(dtype) for y in twin.forward_groups([(x.float(), i) for x, i in groups])]


def twin_inverse(twin, groups, dtype):
    return [o.to(dtype) for o in twin.inverse_groups([(s.float(), i) for s, i in groups])]


def twin_step(twin, groups, dtype):
    ys = twin_forward(twin, groups, dtype)
    return list(zip(twin_inverse(twin, [(y, i) for y, (_, i) in zip(ys, groups)], dtype), ys))


def results_equal(got, want):
    for g, w in zip(got, want):
        if isinstance(g, tuple):
            if not (bits_equal(g[0], w[0]) and bits_equal(g[1], w[1])):
                return False
        elif not bits_equal(g, w):
            return False
    return len(got) == len(want)


# ---------------------------------------------------------------- the C entries
class _Group(ctypes.Structure):
    _fields_ = [("ids", ctypes.c_void_p), ("n", ctypes.c_int), ("T", ctypes.c_long), ("x", ctypes.c_void_p), ("y", ctypes.c_void_p),
                ("out", ctypes.c_void_p)]


def _cabi(pq):
    c = pq._lib.cabi
    vp, i, u = ctypes.c_void_p, ctypes.c_int, ctypes.c_uint
    gp, up = ctypes.POINTER(_Group), ctypes.POINTER(ctypes.c_uint)
    for f in (c.pqmf_stream_pool_analysis_groups_x, c.pqmf_stream_pool_synthesis_groups_x):
        f.argtypes = [gp, i, vp, vp, vp, vp, i, i, i, u, i, up, vp]
        f.restype = ctypes.c_int
    return c


def c_call(pq, mod, pool, groups, direction, dtype, outs=None):
    """pqmf_stream_pool_{analysis,synthesis}_groups_x on (block, ids) groups: (rc, staged, launches, [output]).  Analysis blocks are
    x [n, 1, T] -> y [n, M, T / M]; synthesis blocks s [n, M, F] -> out [n, 1, M F]."""
    c = _cabi(pq)
    m, L = mod.hk.shape
    arr = (_Group * max(len(groups), 1))()
    res = []
    for k, (b, i) in enumerate(groups):
        n = b.shape[0]
        if direction == "analysis":
            T = b.shape[2]
            o = outs[k] if outs else torch.empty(n, m, T // m, dtype=dtype, device="cuda")
            arr[k] = _Group(i.data_ptr(), n, T, b.data_ptr(), o.data_ptr(), None)
        else:
            T = b.shape[2] * m
            o = outs[k] if outs else torch.empty(n, 1, T, dtype=dtype, device="cuda")
            arr[k] = _Group(i.data_ptr(), n, T, None, b.data_ptr(), o.data_ptr())
        res.append(o)
    staged = ctypes.c_uint(0xFFFF)
    launches = pq.launch_count()
    st = torch.cuda.current_stream().cuda_stream
    if direction == "analysis":
        rc = c.pqmf_stream_pool_analysis_groups_x(arr, len(groups), mod.hk.data_ptr(), mod._tables.data_ptr(), pool.xpool.data_ptr(),
                                                  pool.xphase.data_ptr(), pool.capacity, m, L, mod._flags, CODE[dtype], ctypes.byref(staged), st)
    else:
        rc = c.pqmf_stream_pool_synthesis_groups_x(arr, len(groups), mod.hk.data_ptr(), mod._tables.data_ptr(), pool.spool.data_ptr(),
                                                   pool.sphase.data_ptr(), pool.capacity, m, L, mod._flags, CODE[dtype], ctypes.byref(staged), st)
    return rc, staged.value, pq.launch_count() - launches, res


# n_band -> block lengths whose groups each run the streaming Hankel-4 kernels alone (7680 at n_band 16: the largest native block)
NATIVE = {8: (512, 1024, 2048), 16: (512, 2048, 7680), 32: (1024, 2048, 4096)}
SERVER_MIX = ((600, 512), (400, 1024), (250, 2048), (90, 4096))  # n_band 16: each group below 96 tiles alone, in both directions


# ---------------------------------------------------------------- 1. native groups
@pytest.mark.gpu
@pytest.mark.parametrize("m", (8, 16, 32))
@pytest.mark.parametrize("dtype", DTYPES)
def test_native_groups_equal_the_twin(pq, mods, dtype, m):
    """Groups that are native alone: 2 launches per direction through the C entries, 4 for step_groups; bit-equal to the twin and to one
    single-group half step per group."""
    mod = mods(100, m)
    shapes = []
    for T in NATIVE[m]:
        sa, ss = _spt(mod, T)
        assert sa and ss, (m, T)
        shapes.append((MIN_TILES * max(sa, ss) + 5, T))
    assert _joined(mod, shapes, 0) == _joined(mod, shapes, 1) == {0, 1, 2}
    P = sum(n for n, _ in shapes) + 64
    a, b, seq = (pq.StreamPool(mod, P, dtype=dtype), pq.StreamPool(mod, P), pq.StreamPool(mod, P, dtype=dtype))
    ids = _split(P, [n for n, _ in shapes], m)
    for step in range(2):
        groups = [(blocks((n, 1, T), 100 * step + k, dtype), ids[k]) for k, (n, T) in enumerate(shapes)]
        want_y = twin_forward(b, groups, dtype)
        rc, staged, launches, ys = c_call(pq, mod, a, groups, "analysis", dtype)
        assert (rc, staged, launches) == (0, 0, 2), step
        assert results_equal(ys, want_y) and pools_equal(a, b), step
        sgroups = [(y, i) for y, (_, i) in zip(ys, groups)]
        want_o = twin_inverse(b, sgroups, dtype)
        rc, staged, launches, outs = c_call(pq, mod, a, sgroups, "synthesis", dtype)
        assert (rc, staged, launches) == (0, 0, 2), step
        assert results_equal(outs, want_o) and pools_equal(a, b), step
        assert results_equal(list(zip(outs, ys)), [seq.step(x, i) for x, i in groups]), step
    groups = [(blocks((n, 1, T), 7 + k, dtype), ids[k]) for k, (n, T) in enumerate(shapes)]
    launches = pq.launch_count()
    got = a.step_groups(groups)
    assert pq.launch_count() - launches == 4
    assert results_equal(got, twin_step(b, groups, dtype)) and pools_equal(a, b)
    assert results_equal(got, [seq.step(x, i) for x, i in groups])


# ---------------------------------------------------------------- 2. the small-group server mix
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_server_mix_reaches_the_tensor_cores_together(pq, mods, dtype):
    mod = mods(100, 16)
    assert _joined(mod, SERVER_MIX, 0) == _joined(mod, SERVER_MIX, 1) == {0, 1, 2, 3}
    P = 2048
    pool, twin, alone = pq.StreamPool(mod, P, dtype=dtype), pq.StreamPool(mod, P), pq.StreamPool(mod, P, dtype=dtype)
    ids = _split(P, [n for n, _ in SERVER_MIX], 1)
    for step in range(2):
        groups = [(blocks((n, 1, T), 10 * step + k, dtype), ids[k]) for k, (n, T) in enumerate(SERVER_MIX)]
        launches = pq.launch_count()
        got = pool.step_groups(groups)
        assert pq.launch_count() - launches == 4
        assert results_equal(got, twin_step(twin, groups, dtype)) and pools_equal(pool, twin), step
        direct = [alone.step(x, i) for x, i in groups]  # each group alone is below the threshold: the direct form (staged)
        for k, ((o, y), (o_d, y_d)) in enumerate(zip(got, direct)):
            assert not (bits_equal(y, y_d) and bits_equal(o, o_d)), (step, k)


# ---------------------------------------------------------------- 3. steady state across group boundaries
def _oracle_rows(mod, before, src, got, ids, rows, direction, dtype, what):
    """Rows of one group against the float64 streaming oracle (on the widened input) within TOL / 2 plus half an ulp of the dtype."""
    m, length = mod.hk.shape
    hk = mod.hk.cpu().double().numpy()
    xpool, spool, xphase, sphase = before
    half_ulp = 2.0 ** -11 if dtype == torch.float16 else 2.0 ** -8
    for r in rows:
        i = int(ids[r])
        st = O.StreamState(1, m, length)
        st.x_hist = xpool[int(xphase[i]) & 1, i].cpu().double().numpy()[None]
        st.s_hist = spool[int(sphase[i]) & 1, i].cpu().double().numpy()[None]
        st.frames_in, st.frames_out = (int(xphase[i]) >> 1) & 1, (int(sphase[i]) >> 1) & 1
        if direction == "analysis":
            ref = O.stream_analysis(src[r : r + 1, 0].double().cpu().numpy(), hk, st)
            val = got[r : r + 1].double().cpu().numpy()
        else:
            ref = O.stream_synthesis(src[r : r + 1].double().cpu().numpy(), hk, st)
            val = got[r : r + 1, 0].double().cpu().numpy()
        err = np.abs(val - ref) - (TOL / 2 + half_ulp * np.abs(ref) + 2.0 ** -25)
        assert err.max() <= 0, (what, r, float(err.max()))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_steady_state_across_group_boundaries(pq, mods, dtype):
    """About ten tiles per CTA over four groups, an odd tile count and a one-stream last tile in each group; oracle rows on every CTA's first
    three and last tiles and on both sides of every group boundary, in both directions.  A build that loaded the first tile after a group
    switch with the previous group's plan (rebuilding it after the loads) fails here."""
    mod = mods(100, 16)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    grid = sms & ~1
    per_group = (10 * grid) // 4 | 1  # odd
    shapes = [((per_group - 1) * _spt(mod, T)[0] + 1, T) for T in (512, 1024, 2048, 4096)]
    P = sum(n for n, _ in shapes) + 17
    a, b = pq.StreamPool(mod, P, dtype=dtype), pq.StreamPool(mod, P)
    ids = _split(P, [n for n, _ in shapes], 2)

    def picks(d):
        tiles = [_tiles(n, _spt(mod, T)[d]) for n, T in shapes]
        tile0, total = np.cumsum([0] + tiles), sum(tiles)
        ts = set()
        for c in range(grid):
            its = list(range(c, total, grid))
            ts.update(its[:3] + its[-1:])
        for k in range(1, 4):
            ts.update((tile0[k] - 1, tile0[k]))
        rows = {}
        for t in sorted(ts):
            k = int(np.searchsorted(tile0, t, side="right") - 1)
            spt = _spt(mod, shapes[k][1])[d]
            row = (t - tile0[k]) * spt
            rows.setdefault(k, set()).update({row, min(row + spt, shapes[k][0]) - 1})
        return rows

    for step in range(2):
        groups = [(blocks((n, 1, T), 50 + 10 * step + k, dtype), ids[k]) for k, (n, T) in enumerate(shapes)]
        before = _state(a)
        launches = pq.launch_count()
        ys = a.forward_groups(groups)
        assert pq.launch_count() - launches == 2
        assert results_equal(ys, twin_forward(b, groups, dtype)) and pools_equal(a, b), step
        sgroups = [(y, i) for y, (_, i) in zip(ys, groups)]
        launches = pq.launch_count()
        outs = a.inverse_groups(sgroups)
        assert pq.launch_count() - launches == 2
        assert results_equal(outs, twin_inverse(b, sgroups, dtype)) and pools_equal(a, b), step
        if step == 1:
            for k, rows in picks(0).items():
                _oracle_rows(mod, before, groups[k][0], ys[k], ids[k], sorted(rows), "analysis", dtype, ("analysis", k))
            for k, rows in picks(1).items():
                _oracle_rows(mod, before, ys[k], outs[k], ids[k], sorted(rows), "synthesis", dtype, ("synthesis", k))


# ---------------------------------------------------------------- 4. directions that join differently
def _one_direction_mix(mod):
    """Two groups that plan in both directions and reach 96 tiles together in exactly one, or None: a block length whose directions put
    different numbers of streams in a tile, 48 tiles per group in the direction with fewer (96 together) and fewer in the other."""
    for T in range(256, 16385, 256):
        sa, ss = _spt(mod, T)
        if sa and ss and sa != ss:
            shapes = [(48 * min(sa, ss), T), (48 * min(sa, ss), T)]
            assert bool(_joined(mod, shapes, 0)) != bool(_joined(mod, shapes, 1)), (T, sa, ss)
            return shapes
    return None


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_directions_join_differently(pq, mods, dtype):
    """A step joins by each direction's own rule: a bank whose synthesis cannot plan, and (where one exists) a mix that reaches 96 tiles in
    one direction only."""
    for att in (50, 80):
        mod = mods(att, 32)
        assert _spt(mod, 2048)[0] and _spt(mod, 2048)[1] is None, att
        shapes = [(MIN_TILES * _spt(mod, T)[0] // 2 + 3, T) for T in (2048, 4096)]
        assert _joined(mod, shapes, 0) == {0, 1} and _joined(mod, shapes, 1) == set()
        P = sum(n for n, _ in shapes)
        pool, twin = pq.StreamPool(mod, P, dtype=dtype), pq.StreamPool(mod, P)
        ids = _split(P, [n for n, _ in shapes], att)
        for step in range(2):
            groups = [(blocks((n, 1, T), att + step + k, dtype), ids[k]) for k, (n, T) in enumerate(shapes)]
            launches = pq.launch_count()
            got = pool.step_groups(groups)
            assert pq.launch_count() - launches == 2 + 2 * len(shapes), att  # grouped analysis; each synthesis alone (direct form + phase)
            assert results_equal(got, twin_step(twin, groups, dtype)) and pools_equal(pool, twin), (att, step)
    for m in (8, 16, 32):
        mod = mods(100, m)
        shapes = _one_direction_mix(mod)
        if shapes is None:  # both directions put the same number of streams in a tile at every block length they plan
            assert all(sa == ss for sa, ss in (_spt(mod, T) for T in range(256, 16385, 256)) if sa and ss), m
            continue
        P = sum(n for n, _ in shapes)
        pool, twin = pq.StreamPool(mod, P, dtype=dtype), pq.StreamPool(mod, P)
        ids = _split(P, [n for n, _ in shapes], m)
        groups = [(blocks((n, 1, T), m + k, dtype), ids[k]) for k, (n, T) in enumerate(shapes)]
        assert results_equal(pool.step_groups(groups), twin_step(twin, groups, dtype)) and pools_equal(pool, twin), m


# ---------------------------------------------------------------- 5. refusals
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_refused_groups(pq, mods, dtype):
    """48- and 480-sample groups next to joined ones are marked in `staged`; a joined group's half view misaligned by one element refuses
    the whole call with nothing launched; a pool of an n_band-4 module runs every group alone.  Through the op every case equals the twin."""
    mod = mods(100, 16)
    P = 3072
    pool, twin = pq.StreamPool(mod, P, dtype=dtype), pq.StreamPool(mod, P)
    shapes = [(600, 512), (200, 480), (400, 1024), (50, 48), (300, 2048)]
    assert _joined(mod, shapes, 0) == _joined(mod, shapes, 1) == {0, 2, 4}
    ids = _split(P, [n for n, _ in shapes], 3)
    for step in range(2):
        groups = [(blocks((n, 1, T), 30 + 10 * step + k, dtype), i) for k, ((n, T), i) in enumerate(zip(shapes, ids))]
        want_y = twin_forward(twin, groups, dtype)
        rc, staged, launches, ys = c_call(pq, mod, pool, groups, "analysis", dtype)
        assert (rc, staged, launches) == (0, 0b01010, 2), step
        for k in (1, 3):  # what the op does for a staged group
            ys[k] = pool.forward(*groups[k])
        assert results_equal(ys, want_y) and pools_equal(pool, twin), step
        sgroups = [(y, i) for y, i in zip(ys, ids)]
        want_o = twin_inverse(twin, sgroups, dtype)
        rc, staged, launches, outs = c_call(pq, mod, pool, sgroups, "synthesis", dtype)
        assert (rc, staged, launches) == (0, 0b01010, 2), step
        for k in (1, 3):
            outs[k] = pool.inverse(*sgroups[k])
        assert results_equal(outs, want_o) and pools_equal(pool, twin), step
        groups = [(blocks((n, 1, T), 80 + 10 * step + k, dtype), i) for k, ((n, T), i) in enumerate(zip(shapes, ids))]
        assert results_equal(pool.step_groups(groups), twin_step(twin, groups, dtype)) and pools_equal(pool, twin), step
    # a half view one element past an aligned start, in a joined group: the block (analysis) and the sub-bands (synthesis)
    groups = [(blocks((n, 1, T), 90 + k, dtype), i) for k, ((n, T), i) in enumerate(zip(shapes, ids))]
    n, T = shapes[2]
    buf = torch.empty(n * T + 1, dtype=dtype, device="cuda")
    buf[1:].copy_(groups[2][0].reshape(-1))
    groups[2] = (buf[1:].view(n, 1, T), ids[2])
    assert groups[2][0].is_contiguous() and groups[2][0].data_ptr() % 16 != 0
    before = _state(pool)
    rc, _, launches, _ = c_call(pq, mod, pool, groups, "analysis", dtype)
    assert (rc, launches) == (ERR_UNSUPPORTED, 0)
    assert all(torch.equal(u, v) for u, v in zip(_state(pool), before))
    ys = pool.forward_groups(groups)
    assert results_equal(ys, twin_forward(twin, groups, dtype)) and pools_equal(pool, twin)
    sgroups = [(y, i) for y, i in zip(ys, ids)]
    sbuf = torch.empty(ys[4].numel() + 1, dtype=dtype, device="cuda")
    sbuf[1:].copy_(ys[4].reshape(-1))
    sgroups[4] = (sbuf[1:].view(ys[4].shape), ids[4])
    before = _state(pool)
    rc, _, launches, _ = c_call(pq, mod, pool, sgroups, "synthesis", dtype)
    assert (rc, launches) == (ERR_UNSUPPORTED, 0)
    assert all(torch.equal(u, v) for u, v in zip(_state(pool), before))
    assert results_equal(pool.inverse_groups(sgroups), twin_inverse(twin, sgroups, dtype)) and pools_equal(pool, twin)
    # n_band 4: no streaming Hankel-4 kernels; every group alone, refused by its single-group entry and staged by the op
    mod4 = mods(100, 4)
    pool4, twin4 = pq.StreamPool(mod4, 2000, dtype=dtype), pq.StreamPool(mod4, 2000)
    shapes4 = [(600, 512), (400, 1024)]
    ids4 = _split(2000, [n for n, _ in shapes4], 4)
    groups = [(blocks((n, 1, T), 60 + k, dtype), i) for k, ((n, T), i) in enumerate(zip(shapes4, ids4))]
    rc, staged, launches, _ = c_call(pq, mod4, pool4, groups, "analysis", dtype)
    assert (rc, staged, launches) == (0, 0b11, 0)
    assert results_equal(pool4.step_groups(groups), twin_step(twin4, groups, dtype)) and pools_equal(pool4, twin4)


# ---------------------------------------------------------------- 6. fp16 overflow
@pytest.mark.gpu
def test_fp16_overflow(pq, mods):
    """Sub-bands near the fp16 maximum reconstruct past it in a grouped inverse: +-inf exactly where .to(float16) of the fp32 result gives
    it."""
    mod = mods(100, 16)
    P = 2048
    pool, twin = pq.StreamPool(mod, P, dtype=torch.float16), pq.StreamPool(mod, P)
    ids = _split(P, [n for n, _ in SERVER_MIX], 6)
    g = torch.Generator(device="cuda").manual_seed(6)
    n_inf = 0
    for k in range(2):
        sgroups = [((6e4 * torch.randn(n, 16, T // 16, device="cuda", generator=g)).clamp_(-65504, 65504).half(), ids[j])
                   for j, (n, T) in enumerate(SERVER_MIX)]
        launches = pq.launch_count()
        outs = pool.inverse_groups(sgroups)
        assert pq.launch_count() - launches == 2
        assert results_equal(outs, twin_inverse(twin, sgroups, torch.float16)) and pools_equal(pool, twin), k
        n_inf += sum(int(torch.isinf(o).sum()) for o in outs)
    assert n_inf > 1000


# ---------------------------------------------------------------- 7. a seeded schedule
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_seeded_schedule_over_a_pool(pq, mods, dtype):
    """Twelve calls over a pool of 4096 mixing step_groups, forward_groups, inverse_groups, step, step_pcm16, step_groups_pcm16 and resets,
    with a dead CUDA id in one group (zeros out, no state touched); unlisted streams keep both halves and their phase words."""
    P, m = 4096, 16
    mod = mods(100, m)
    pool, twin = pq.StreamPool(mod, P, dtype=dtype), pq.StreamPool(mod, P)
    rng = np.random.default_rng(13)
    lengths = (48, 256, 480, 512, 1024, 2048, 4096)
    kinds = ("step_groups", "forward_groups", "inverse_groups", "step", "step_groups_pcm16", "step_groups",
             "pcm16", "step_groups", "forward_groups", "inverse_groups", "step_groups", "step")
    for k, kind in enumerate(kinds):
        if k in (4, 9):
            gone = rng.choice(P, 500, replace=False).tolist()
            pool.reset(gone)
            twin.reset(gone)
        G = int(rng.integers(2, 9)) if "groups" in kind else 1
        n_all = int(rng.integers(G, 3000))
        chosen = rng.choice(P, n_all, replace=False)
        parts = np.split(chosen, np.sort(rng.choice(np.arange(1, n_all), G - 1, replace=False))) if G > 1 else [chosen]
        lens = [int(rng.choice(lengths)) for _ in parts]
        ids = [torch.from_numpy(p.astype(np.int32)).cuda() for p in parts]
        dead = k == 5
        if dead:  # one dead row in the first group: an id outside [0, P)
            ids[0] = torch.cat([ids[0], torch.tensor([P + 3], dtype=torch.int32, device="cuda")])
        before = _state(pool)
        if kind in ("step_groups", "forward_groups", "step"):
            groups = [(blocks((i.numel(), 1, T), 1000 * k + j, dtype), i) for j, (i, T) in enumerate(zip(ids, lens))]
            if kind == "step_groups":
                got, want = pool.step_groups(groups), twin_step(twin, groups, dtype)
            elif kind == "forward_groups":
                got, want = pool.forward_groups(groups), twin_forward(twin, groups, dtype)
            else:
                got, want = [pool.step(*groups[0])], twin_step(twin, groups[:1], dtype)
        elif kind == "inverse_groups":
            groups = [(blocks((i.numel(), m, T // m), 1000 * k + j, dtype), i) for j, (i, T) in enumerate(zip(ids, lens))]
            got, want = pool.inverse_groups(groups), twin_inverse(twin, groups, dtype)
        else:  # PCM calls behave as on a float32 pool: the state is shared
            gen = torch.Generator(device="cuda").manual_seed(k)
            groups = [((8000 * torch.randn(i.numel(), T, 1, device="cuda", generator=gen)).round().clamp(-32768, 32767).to(torch.int16), i)
                      for i, T in zip(ids, lens)]
            got = pool.step_groups_pcm16(groups) if kind == "step_groups_pcm16" else [pool.step_pcm16(*groups[0])]
            want = twin.step_groups_pcm16(groups) if kind == "step_groups_pcm16" else [twin.step_pcm16(*groups[0])]
            assert all(torch.equal(o, o_r) and torch.equal(y, y_r) for (o, y), (o_r, y_r) in zip(got, want)), (k, kind)
            got = want = []
        assert results_equal(got, want), (k, kind)
        if dead:
            o, y = got[0]
            assert not y[-1].float().any() and not o[-1].float().any()
        assert pools_equal(pool, twin), (k, kind)
        listed = torch.cat([i[(i >= 0) & (i < P)] for i in ids]).long()
        rest = torch.ones(P, dtype=torch.bool, device="cuda")
        rest[listed] = False
        for now, then in zip(_state(pool), before):
            assert torch.equal(now[:, rest] if now.dim() > 1 else now[rest], then[:, rest] if then.dim() > 1 else then[rest]), (k, kind)


# ---------------------------------------------------------------- 8. CUDA graph
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_one_graph_replays_grouped_half_steps(pq, mods, dtype):
    mod = mods(100, 16)
    P = 2048
    graph_pool, eager = pq.StreamPool(mod, P, dtype=dtype), pq.StreamPool(mod, P, dtype=dtype)
    rng = np.random.default_rng(3)
    pre = torch.from_numpy(rng.choice(P, P // 3, replace=False).astype(np.int32)).cuda()  # mixed parities, identically on both pools
    xpre = blocks((pre.numel(), 1, 48), 1, dtype)
    graph_pool.step(xpre, pre)
    eager.step(xpre, pre)
    static = [(torch.zeros(n, 1, T, dtype=dtype, device="cuda"), torch.arange(r0, r0 + n, dtype=torch.int32, device="cuda"))
              for (n, T), r0 in zip(SERVER_MIX, np.cumsum([0] + [n for n, _ in SERVER_MIX])[:-1].tolist())]
    warm = pq.StreamPool(mod, P, dtype=dtype)  # first launches set the kernels' shared-memory limits: not inside a capture
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
            x = blocks((n, 1, T), 300 + 10 * k + r0 % 7, dtype)
            sx.copy_(x)
            si.copy_(perm[r0 : r0 + n])
            eager_groups.append((x, perm[r0 : r0 + n]))
            r0 += n
        graph.replay()
        assert results_equal(g_res, eager.step_groups(eager_groups)) and pools_equal(graph_pool, eager), k


# ---------------------------------------------------------------- 9. C outputs inside guard words
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_write_guards(pq, mods, dtype):
    """The C entries write only inside every group's y and out, joined and staged groups alike."""
    mod = mods(100, 16)
    P, margin = 1300, 1024
    shapes = SERVER_MIX[:2] + ((50, 48), (60, 480))
    pool, ref = pq.StreamPool(mod, P, dtype=dtype), pq.StreamPool(mod, P, dtype=dtype)
    ids = _split(P, [n for n, _ in shapes], 5)
    bufs = []

    def guarded(n):
        buf = torch.full((n + 2 * margin,), GUARD, dtype=torch.int16, device="cuda")
        bufs.append(buf)
        return buf[margin : margin + n].view(dtype)

    groups = [(blocks((n, 1, T), k, dtype), ids[k]) for k, (n, T) in enumerate(shapes)]
    ys = [guarded(n * T).view(n, 16, T // 16) for n, T in shapes]
    rc, staged, launches, _ = c_call(pq, mod, pool, groups, "analysis", dtype, ys)
    assert (rc, staged, launches) == (0, 0b1100, 2)
    for k in (2, 3):
        ys[k].copy_(pool.forward(*groups[k]))
    outs = [guarded(n * T).view(n, 1, T) for n, T in shapes]
    sgroups = [(y, i) for y, i in zip(ys, ids)]
    rc, staged, launches, _ = c_call(pq, mod, pool, sgroups, "synthesis", dtype, outs)
    assert (rc, staged, launches) == (0, 0b1100, 2)
    for k in (2, 3):
        outs[k].copy_(pool.inverse(*sgroups[k]))
    torch.cuda.synchronize()
    for b in bufs:
        assert (b[:margin] == GUARD).all() and (b[-margin:] == GUARD).all()
    assert results_equal(list(zip(outs, ys)), ref.step_groups(groups)) and pools_equal(pool, ref)


# ---------------------------------------------------------------- 10. errors
@pytest.mark.gpu
def test_group_half_errors(pq, mods):
    mod = mods(100, 16)
    for dtype, other, name in ((torch.bfloat16, torch.float32, "Float"), (torch.float16, torch.bfloat16, "BFloat16")):
        pool = pq.StreamPool(mod, 64, dtype=dtype)
        x = torch.zeros(3, 1, 256, dtype=dtype, device="cuda")
        s = torch.zeros(3, 16, 16, dtype=dtype, device="cuda")
        n0 = pq.launch_count()
        with pytest.raises(RuntimeError, match=name):
            pool.forward_groups([(x, [0, 1, 2]), (x.to(other), [3, 4, 5])])
        with pytest.raises(RuntimeError, match=name):
            pool.inverse_groups([(s, [0, 1, 2]), (s.to(other), [3, 4, 5])])
        with pytest.raises(RuntimeError, match=name):  # the op names the pool's dtype too, before anything is launched
            torch.ops.pqmf_b200.stream_pool_analysis_groups_x([x, x.to(other)], mod.hk.float(), mod._tables, pool.xpool, pool.xphase,
                                                              [torch.arange(3, dtype=torch.int32, device="cuda")] * 2, dtype, mod._flags)
        with pytest.raises(RuntimeError, match="not differentiable"):
            pool.inverse_groups([(s.clone().requires_grad_(), [0, 1, 2])])
        with pytest.raises(RuntimeError, match="not differentiable"):
            pool.forward_groups([(x.clone().requires_grad_(), [0, 1, 2])])
        with pytest.raises(ValueError, match="at most 8"):
            pool.forward_groups([(x, [3 * k, 3 * k + 1, 3 * k + 2]) for k in range(9)])
        with pytest.raises(RuntimeError, match="at most 8"):
            torch.ops.pqmf_b200.stream_pool_synthesis_groups_x([s] * 9, mod.hk.float(), mod._tables, pool.spool, pool.sphase,
                                                               [torch.arange(3, dtype=torch.int32, device="cuda")] * 9, dtype, mod._flags)
        with pytest.raises(ValueError, match="across all groups"):
            pool.step_groups([(x, [0, 1, 2]), (x, [3, 4, 0])])
        with pytest.raises(RuntimeError, match="float32, float16 or bfloat16"):
            torch.ops.pqmf_b200.stream_pool_analysis_groups_x([], mod.hk.float(), mod._tables, pool.xpool, pool.xphase, [], torch.float64,
                                                              mod._flags)
        assert pq.launch_count() == n0
        assert (pool.xphase == 0).all() and (pool.sphase == 0).all() and not pool.xpool.any() and not pool.spool.any()
        assert pool.step_groups([]) == [] and pool.forward_groups([(x[:0], [])])[0].shape == (0, 16, 16)
        assert pool.inverse_groups([(s[:0], [])])[0].dtype == dtype
        assert pq.launch_count() == n0


# ---------------------------------------------------------------- 11. C argument checks (no GPU)
def test_group_half_cabi_argument_checks_happen_before_any_cuda_call(pq):
    """The grouped _x entries validate on the host and return PQMF_ERR_ARG (or 0 when there are no rows) without touching a device."""
    c = _cabi(pq)
    an, sy = c.pqmf_stream_pool_analysis_groups_x, c.pqmf_stream_pool_synthesis_groups_x
    fake = 4096  # never dereferenced: every call below fails a host check or has no rows

    def groups(*specs):
        arr = (_Group * max(len(specs), 1))()
        for k, (n, T, ptrs) in enumerate(specs):
            q = fake if ptrs else None
            arr[k] = _Group(q, n, T, q, q, q)
        return arr

    def call(f, arr, G, code, P=64, M=16, L=512, pools=True, staged=True):
        p = fake if pools else None
        mask = ctypes.c_uint(77)
        rc = f(arr, G, fake, None, p, p, P, M, L, 0, code, ctypes.byref(mask) if staged else None, None)
        return rc, mask.value

    for f in (an, sy):
        for code in (DT_F16, DT_BF16, DT_F32):
            assert call(f, groups(), 0, code) == (0, 0)                                    # G == 0
            assert call(f, groups((0, 512, False), (0, 2048, False)), 2, code) == (0, 0)   # all empty
            assert call(f, groups((0, 512, False)), 1, code, pools=False) == (0, 0)        # all empty, no pools
            assert call(f, groups(), -1, code)[0] == ERR_ARG                               # G < 0
            assert call(f, groups(*[(1, 512, True)] * 9), 9, code)[0] == ERR_ARG           # G > 8
            assert call(f, None, 2, code)[0] == ERR_ARG                                    # no descriptors
            assert call(f, groups((40, 512, True), (30, 512, True)), 2, code)[0] == ERR_ARG  # more rows than P
            assert call(f, groups((4, 520, True), (4, 512, True)), 2, code)[0] == ERR_ARG  # T % M != 0
            assert call(f, groups((4, 0, True), (4, 512, True)), 2, code)[0] == ERR_ARG    # T == 0
            assert call(f, groups((4, 512, False), (4, 512, True)), 2, code)[0] == ERR_ARG  # null pointers in a non-empty group
            assert call(f, groups((-1, 512, True)), 1, code)[0] == ERR_ARG                 # n < 0
            assert call(f, groups((4, 512, True)), 1, code, P=0)[0] == ERR_ARG             # P < 1
            assert call(f, groups((4, 512, True), (4, 512, True)), 2, code, pools=False)[0] == ERR_ARG  # null pool
            assert call(f, groups((4, 512, True)), 1, code, staged=False)[0] == ERR_ARG    # null staged
            assert call(f, groups(), 0, code, staged=False)[0] == ERR_ARG                  # null staged, no groups
        for code in (-1, 3, 7):                                                            # an unknown dtype, whatever else the call holds
            assert call(f, groups(), 0, code)[0] == ERR_ARG
            assert call(f, groups((0, 512, False)), 1, code)[0] == ERR_ARG
    # PQMF_DTYPE_F32 is the _f32 grouped entry: its own return codes
    for f, g in ((an, c.pqmf_stream_pool_analysis_groups_f32), (sy, c.pqmf_stream_pool_synthesis_groups_f32)):
        g.restype = ctypes.c_int
        g.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
                      ctypes.c_int, ctypes.c_uint, ctypes.c_void_p]
        for arr, G in ((groups(), 0), (groups((0, 512, False)), 1), (groups((40, 512, True), (30, 512, True)), 2),
                       (groups((4, 520, True)), 1), (groups((4, 512, False)), 1), (groups(*[(1, 512, True)] * 9), 9)):
            want = g(ctypes.cast(arr, ctypes.c_void_p), G, fake, None, fake, fake, 64, 16, 512, 0, None)
            assert call(f, arr, G, DT_F32)[0] == want
