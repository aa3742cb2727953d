"""Half-precision stream pools: StreamPool(mod, P, dtype=torch.float16 / torch.bfloat16).

Every call on a half pool must give, per row, the bits of a twin float32 pool: forward(x) = twin.forward(x.float()).to(dtype),
inverse(s) = twin.inverse(s.float()).to(dtype), step(x) = (inverse(y), y) with y = forward(x) -- the synthesis reads the ROUNDED
sub-bands -- with pool buffers and phase words equal to the twin's, whether the call runs the streaming Hankel-4 kernels with half loads
and stores or is staged.  The C entries (pqmf_stream_pool_*_x) must run natively exactly where the float32 pool call runs those kernels,
and refuse every other call before launching anything.  The last test needs no GPU: it checks the C entries' argument validation."""
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
N_SM = 148
GUARD = 0x7DAD  # guard half word: a NaN in bf16 and fp16 that no kernel writes


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


def _cabi(pq):
    c = pq._lib.cabi
    vp, i, lg, u = ctypes.c_void_p, ctypes.c_int, ctypes.c_long, ctypes.c_uint
    c.pqmf_stream_pool_analysis_x.argtypes = [vp] * 6 + [i, vp, i, lg, i, i, u, i, vp]
    c.pqmf_stream_pool_synthesis_x.argtypes = [vp] * 6 + [i, vp, i, lg, i, i, u, i, vp]
    c.pqmf_stream_pool_step_x.argtypes = [vp] * 9 + [i, vp, i, lg, i, i, u, i, vp]
    for f in ("analysis", "synthesis", "step"):
        getattr(c, f"pqmf_stream_pool_{f}_x").restype = ctypes.c_int
    return c


# ---------------------------------------------------------------- the float32 pool's streaming plan (h4_*_stream_plan), host arithmetic
def _taps(flags):
    return 32 * ((flags >> 8) & 0xF), 32 * ((flags >> 12) & 0x1F)


def _hist_rows(mod):
    """history rows in front of every block, (analysis, synthesis); the banks used here have a plan in both directions"""
    m, L = mod.hk.shape
    jlo, kt = _taps(mod._flags)
    a = -(-(L - jlo) // 64)
    frames = -(-((jlo + kt) // m) * m // 64) * 64 // m
    return a, frames * m // 64


def _spt(T, hrows):
    pitch = (T // 64 + hrows + 3) & ~3
    return 128 // pitch if pitch <= 128 else 0


def native(mod, B, T):
    """the float32 pool call of B rows of T samples runs the streaming Hankel-4 kernels in both directions"""
    m, L = mod.hk.shape
    if T % 256 or T < L:
        return False
    return all(_spt(T, h) >= 1 and -(-B // _spt(T, h)) >= 96 for h in _hist_rows(mod))


def largest_native(mod):
    return max(T for T in range(256, 16385, 256) if native(mod, 1 << 20, T))


# ---------------------------------------------------------------- helpers
def blocks(shape, seed, dtype, scale=0.5):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (scale * torch.randn(shape, device="cuda", generator=g)).clamp_(-1, 1).to(dtype)


def pools_equal(a, b):
    return all(torch.equal(u, v) for u, v in zip((a.xpool, a.spool, a.xphase, a.sphase), (b.xpool, b.spool, b.xphase, b.sphase)))


def twin_step(twin, x, ids, dtype):
    """the contract of a half step on a float32 pool: analysis of the widened block, rounding, synthesis of the rounded sub-bands"""
    y = twin.forward(x.float(), ids).to(dtype)
    return twin.inverse(y.float(), ids).to(dtype), y


def check_calls(pool, twin, kinds, B, T, seed, dtype, ids_of=None):
    """run `kinds` ("step", "split", "3frames") on pool and twin; outputs and pools bit-equal after every call"""
    m = pool.mod.n_band
    for k, kind in enumerate(kinds):
        t = 3 * m if kind == "3frames" else T
        ids = ids_of(k) if ids_of else torch.arange(B, dtype=torch.int32, device="cuda")
        x = blocks((B, 1, t), seed + k, dtype)
        if kind == "split":
            y = pool.forward(x, ids)
            assert torch.equal(y, twin.forward(x.float(), ids).to(dtype)) and pools_equal(pool, twin), (k, kind)
            s = blocks((B, m, t // m), seed + 50 + k, dtype)
            out = pool.inverse(s, ids)
            assert torch.equal(out, twin.inverse(s.float(), ids).to(dtype)) and pools_equal(pool, twin), (k, kind)
            continue
        out, y = pool.step(x, ids)
        out_r, y_r = twin_step(twin, x, ids, dtype)
        assert y.dtype == dtype and out.dtype == dtype
        assert torch.equal(y, y_r) and torch.equal(out, out_r) and pools_equal(pool, twin), (k, kind)


def c_route(pq, mod, B, T, dtype, offset=0):
    """(return code, launches) of the three C entries on B rows of T samples (ids = arange, P = B + 3); offset: the half buffers start
    that many elements past a 256-byte boundary.  Refused calls must launch nothing and write nothing."""
    c = _cabi(pq)
    m, L = mod.hk.shape
    hk, tab, fl = mod.hk.float().contiguous(), mod._tables, mod._flags
    st = torch.cuda.current_stream().cuda_stream
    P = B + 3
    xb = blocks((B * T + 64,), B + T, dtype)
    x = xb[offset:offset + B * T]
    yb = torch.zeros(B * T + 64, dtype=dtype, device="cuda")
    y = yb[offset:offset + B * T]
    ob = torch.zeros(B * T + 64, dtype=dtype, device="cuda")
    out = ob[offset:offset + B * T]
    xpool, spool = torch.randn(2, P, L, device="cuda"), torch.randn(2, P, L, device="cuda")
    xph = torch.randint(0, 4, (P,), dtype=torch.int32, device="cuda")
    sph = torch.randint(0, 4, (P,), dtype=torch.int32, device="cuda")
    ids = torch.arange(B, dtype=torch.int32, device="cuda")
    code = CODE[dtype]
    rcs, touched = {}, {}
    for name in ("analysis", "synthesis", "step"):
        snap = [t.clone() for t in (yb, ob, xpool, spool, xph, sph)]
        n0 = pq.launch_count()
        if name == "analysis":
            rc = c.pqmf_stream_pool_analysis_x(x.data_ptr(), y.data_ptr(), hk.data_ptr(), tab.data_ptr(), xpool.data_ptr(), xph.data_ptr(), P,
                                               ids.data_ptr(), B, T, m, L, fl, code, st)
        elif name == "synthesis":
            rc = c.pqmf_stream_pool_synthesis_x(x.data_ptr(), out.data_ptr(), hk.data_ptr(), tab.data_ptr(), spool.data_ptr(), sph.data_ptr(), P,
                                                ids.data_ptr(), B, T // m, m, L, fl, code, st)
        else:
            rc = c.pqmf_stream_pool_step_x(x.data_ptr(), y.data_ptr(), out.data_ptr(), hk.data_ptr(), tab.data_ptr(), xpool.data_ptr(), xph.data_ptr(),
                                           spool.data_ptr(), sph.data_ptr(), P, ids.data_ptr(), B, T, m, L, fl, code, st)
        rcs[name] = (rc, pq.launch_count() - n0)
        torch.cuda.synchronize()
        touched[name] = not all(torch.equal(a, b) for a, b in zip(snap, (yb, ob, xpool, spool, xph, sph)))
    return rcs, touched


NATIVE = {"analysis": (0, 2), "synthesis": (0, 2), "step": (0, 3)}
REFUSED = {"analysis": (ERR_UNSUPPORTED, 0), "synthesis": (ERR_UNSUPPORTED, 0), "step": (ERR_UNSUPPORTED, 0)}


def check_c_route(pq, mod, B, T, dtype, want_native, offset=0):
    rcs, touched = c_route(pq, mod, B, T, dtype, offset)
    if want_native:
        assert rcs == NATIVE, (B, T, rcs)
    else:
        assert rcs == REFUSED and not any(touched.values()), (B, T, offset, rcs, touched)


# ---------------------------------------------------------------- 1. block geometries of the float32 pool's plan
GEOMETRY_CASES = ["T=L", "T=2048", "T=max", "T=max+256", "tiles=95", "tiles=96", "tiles=97"]


def geometry_shape(mod, case):
    L = mod.hk.shape[1]
    t_max = largest_native(mod)
    T = {"T=L": max(L, 256), "T=max": t_max, "T=max+256": t_max + 256}.get(case, 2048)
    spt = min(_spt(T, h) for h in _hist_rows(mod)) or 1
    n_tiles = int(case.split("=")[1]) if case.startswith("tiles") else 101
    return (spt * (n_tiles - 1) + 1 if spt > 1 else n_tiles), T


@pytest.mark.gpu
@pytest.mark.parametrize("case", GEOMETRY_CASES)
@pytest.mark.parametrize("m", [8, 16, 32])
@pytest.mark.parametrize("dtype", DTYPES)
def test_block_geometry(pq, mods, dtype, m, case):
    """Native on the plan's geometries (partial last tiles), refused one block row past the largest native block and one tile below the
    threshold; every call bit-equal to the float32 twin, with the 3-frame block (staged) putting the native calls on both parities."""
    mod = mods(100, m)
    B, T = geometry_shape(mod, case)
    want = case not in ("T=max+256", "tiles=95")
    assert native(mod, B, T) == want, (B, T)
    check_c_route(pq, mod, B, T, dtype, want)
    pool, twin = pq.StreamPool(mod, B + 7, dtype=dtype), pq.StreamPool(mod, B + 7)
    perm = lambda k: torch.randperm(B + 7, device="cuda")[:B].to(torch.int32)  # noqa: E731
    check_calls(pool, twin, ("step", "3frames", "split", "step"), B, T, m + T, dtype, ids_of=perm)


# ---------------------------------------------------------------- 2. steady state: ~10 tiles per CTA against the float64 oracle
@pytest.mark.gpu
@pytest.mark.parametrize("m", [8, 16, 32])
@pytest.mark.parametrize("dtype", DTYPES)
def test_steady_state(pq, mods, dtype, m):
    """4096 streams x 2048 samples: every row bit-equal to the twin; the first row of the tile each CTA runs first and last, and the
    partial last tile, followed through the float64 streaming oracle (on the widened block and the rounded sub-bands) within TOL / 2 plus
    half an ulp of the dtype."""
    B, T = 4096, 2048
    mod = mods(100, m)
    L = mod.hk.shape[1]
    spt = min(_spt(T, h) for h in _hist_rows(mod))
    n_tiles = -(-B // spt)
    assert native(mod, B, T) and n_tiles >= 9 * N_SM
    check_c_route(pq, mod, B, T, dtype, True)
    last = {c: c + N_SM * ((n_tiles - 1 - c) // N_SM) for c in range(N_SM)}
    rows = sorted({spt * c for c in range(N_SM)} | {spt * t for t in last.values()} | set(range((n_tiles - 1) * spt, B)))
    P = B + 40
    pool, twin = pq.StreamPool(mod, P, dtype=dtype), pq.StreamPool(mod, P)
    ids = torch.randperm(P, device="cuda")[:B].to(torch.int32)
    hk = mod.hk.cpu().double().numpy()
    st = O.StreamState(len(rows), m, L)
    half_ulp = 2.0 ** -11 if dtype == torch.float16 else 2.0 ** -8
    for k in range(3):
        x = blocks((B, 1, T), 30 + k, dtype)
        out, y = pool.step(x, ids)
        out_r, y_r = twin_step(twin, x, ids, dtype)
        assert torch.equal(y, y_r) and torch.equal(out, out_r) and pools_equal(pool, twin), k
        y64 = O.stream_analysis(x[rows, 0].double().cpu().numpy(), hk, st)
        o64 = O.stream_synthesis(y[rows].double().cpu().numpy(), hk, st)
        for got, ref in ((y[rows].double().cpu().numpy(), y64), (out[rows, 0].double().cpu().numpy(), o64)):
            err = np.abs(got - ref) - (TOL / 2 + half_ulp * np.abs(ref) + 2.0 ** -25)
            assert err.max() <= 0, (k, float(err.max()))


# ---------------------------------------------------------------- 3. staged routes: refused by the C entry, staged by the op
STAGED = {"few streams": (100, 16, 7, 2048, 0), "n_band 4": (100, 4, 400, 2048, 0), "split bank": (110, 32, 400, 2048, 0),
          "misaligned": (100, 16, 400, 2048, 1), "3 frames": (100, 16, 400, 48, 0)}


@pytest.mark.gpu
@pytest.mark.parametrize("route", list(STAGED))
@pytest.mark.parametrize("dtype", DTYPES)
def test_staged_routes(pq, mods, dtype, route):
    att, m, B, T, offset = STAGED[route]
    mod = mods(att, m)
    if route == "split bank":
        assert mod._flags & pq._lib.PQMF_FLAG_H4_SPLIT
    if route == "3 frames":
        T = 3 * m
    check_c_route(pq, mod, B, T, dtype, False, offset)
    pool, twin = pq.StreamPool(mod, B + 2, dtype=dtype), pq.StreamPool(mod, B + 2)
    for k in range(3):
        x = blocks((B * T + 16,), 5 * k + m, dtype)
        x = x[offset:offset + B * T].view(B, 1, T)  # a contiguous view `offset` elements past an aligned address
        assert x.is_contiguous() and (x.data_ptr() % 16 != 0) == (offset != 0)
        ids = torch.randperm(B + 2, device="cuda")[:B].to(torch.int32)
        out, y = pool.step(x, ids)
        out_r, y_r = twin_step(twin, x, ids, dtype)
        assert torch.equal(y, y_r) and torch.equal(out, out_r) and pools_equal(pool, twin), (route, k)


# ---------------------------------------------------------------- 4. fp16 overflow
@pytest.mark.gpu
@pytest.mark.parametrize("m", [8, 32])
def test_fp16_overflow(pq, mods, m):
    """Sub-bands near the fp16 maximum reconstruct past it: +-inf exactly where torch's .to(float16) of the fp32 result gives it."""
    mod = mods(100, m)
    B, T = 400, 2048
    assert native(mod, B, T)
    pool, twin = pq.StreamPool(mod, B, dtype=torch.float16), pq.StreamPool(mod, B)
    ids = torch.arange(B, dtype=torch.int32, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(m)
    n_inf = 0
    for k in range(3):
        s = (6e4 * torch.randn(B, m, T // m, device="cuda", generator=g)).clamp_(-65504, 65504).half()
        out = pool.inverse(s, ids)
        want = twin.inverse(s.float(), ids).half()
        assert torch.equal(out, want) and pools_equal(pool, twin), k
        n_inf += int(torch.isinf(out).sum())
        x = (6e4 * torch.randn(B, 1, T, device="cuda", generator=g)).clamp_(-65504, 65504).half()
        y = pool.forward(x, ids)
        assert torch.equal(y, twin.forward(x.float(), ids).half()) and pools_equal(pool, twin), k
    assert n_inf > 1000


# ---------------------------------------------------------------- 5. a seeded schedule of every call kind
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_schedule(pq, mods, dtype):
    """12 calls over a pool of 4096: steps, split directions, PCM steps, resets, native and staged shapes, random subsets and orders, and a
    dead CUDA id (zeros out, no state touched).  After every call outputs, pools and phase words equal the twin's; unlisted streams are
    unchanged."""
    P, m = 4096, 16
    mod = mods(100, m)
    pool, twin = pq.StreamPool(mod, P, dtype=dtype), pq.StreamPool(mod, P)
    rng = np.random.default_rng(12)
    schedule = [("step", 4096, 2048), ("forward", 1500, 2048), ("inverse", 1500, 2048), ("pcm", 600, 2048), ("step", 2000, 48),
                ("reset", 700, 0), ("step", 1200, 4096), ("dead", 900, 2048), ("forward", 40, 2048), ("inverse", 3000, 1024),
                ("pcm", 300, 48), ("step", 4096, 2048)]
    for k, (kind, n, T) in enumerate(schedule):
        ids_np = rng.choice(P, n, replace=False).astype(np.int32)
        if kind == "reset":
            pool.reset(ids_np.tolist())
            twin.reset(ids_np.tolist())
            assert pools_equal(pool, twin)
            continue
        dead = None
        if kind == "dead":
            dead = int(rng.integers(n))
            ids_np[dead] = P + 5
        ids = torch.from_numpy(ids_np).cuda()
        before = [t.clone() for t in (pool.xpool, pool.spool, pool.xphase, pool.sphase)]
        if kind in ("step", "dead"):
            x = blocks((n, 1, T), 100 + k, dtype)
            out, y = pool.step(x, ids if k % 2 else ids_np.tolist() if dead is None else ids)
            out_r, y_r = twin_step(twin, x, ids, dtype)
            assert torch.equal(y, y_r) and torch.equal(out, out_r), k
            if dead is not None:
                assert not y[dead].any() and not out[dead].any()
        elif kind == "forward":
            x = blocks((n, 1, T), 100 + k, dtype)
            assert torch.equal(pool.forward(x, ids), twin.forward(x.float(), ids).to(dtype)), k
        elif kind == "inverse":
            s = blocks((n, m, T // m), 100 + k, dtype)
            assert torch.equal(pool.inverse(s, ids), twin.inverse(s.float(), ids).to(dtype)), k
        else:  # PCM calls behave as on a float32 pool: the state is shared
            g = torch.Generator(device="cuda").manual_seed(k)
            pcm = (8000 * torch.randn(n, T, 1, device="cuda", generator=g)).round().clamp(-32768, 32767).to(torch.int16)
            a, b = pool.step_pcm16(pcm, ids), twin.step_pcm16(pcm, ids)
            assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]), k
        assert pools_equal(pool, twin), k
        rest = torch.ones(P, dtype=torch.bool, device="cuda")
        live = ids.long()[(ids >= 0) & (ids < P)]
        rest[live] = False
        for u, v in zip((pool.xpool, pool.spool), before[:2]):
            assert torch.equal(u[:, rest], v[:, rest]), k
        for u, v in zip((pool.xphase, pool.sphase), before[2:]):
            assert torch.equal(u[rest], v[rest]), k


# ---------------------------------------------------------------- 6. staged grouped calls
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_grouped_calls_staged(pq, mods, dtype):
    """step_groups / forward_groups / inverse_groups on a half pool: the twin's grouped calls on the widened groups, rounded, the step's
    synthesis reading the rounded sub-bands."""
    m, P = 16, 3000
    mod = mods(100, m)
    pool, twin = pq.StreamPool(mod, P, dtype=dtype), pq.StreamPool(mod, P)
    rng = np.random.default_rng(6)
    sizes = ((300, 2048), (200, 1024), (90, 48), (400, 4096))
    for k in range(3):
        ids = np.split(rng.choice(P, sum(n for n, _ in sizes), replace=False).astype(np.int32), np.cumsum([n for n, _ in sizes])[:-1])
        ids = [torch.from_numpy(i).cuda() for i in ids]
        xs = [blocks((n, 1, T), 10 * k + j, dtype) for j, (n, T) in enumerate(sizes)]
        got = pool.step_groups(list(zip(xs, ids)))
        ys_r = [y.to(dtype) for y in twin.forward_groups([(x.float(), i) for x, i in zip(xs, ids)])]
        outs_r = [o.to(dtype) for o in twin.inverse_groups([(y.float(), i) for y, i in zip(ys_r, ids)])]
        for (out, y), out_r, y_r in zip(got, outs_r, ys_r):
            assert out.dtype == dtype and torch.equal(y, y_r) and torch.equal(out, out_r), k
        assert pools_equal(pool, twin), k
        ys = pool.forward_groups(list(zip(xs, ids)))
        assert all(torch.equal(y, r.to(dtype)) for y, r in zip(ys, twin.forward_groups([(x.float(), i) for x, i in zip(xs, ids)])))
        outs = pool.inverse_groups(list(zip(ys, ids)))
        assert all(torch.equal(o, r.to(dtype)) for o, r in zip(outs, twin.inverse_groups([(y.float(), i) for y, i in zip(ys, ids)])))
        assert pools_equal(pool, twin), k


# ---------------------------------------------------------------- 7. a module cast to bfloat16
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_pool_of_cast_module(pq, dtype):
    """The pool's dtype is independent of the module's: a .to(torch.bfloat16) module's pool equals a float32 pool of the same module."""
    mod = pq.CachedPQMF(100, 16).cuda().to(torch.bfloat16)
    assert mod.hk.dtype == torch.bfloat16
    B, T = 400, 2048
    assert native(mod, B, T)
    pool, twin = pq.StreamPool(mod, B, dtype=dtype), pq.StreamPool(mod, B)
    assert pool.dtype == dtype and pool.xpool.dtype == torch.float32 and pool.spool.dtype == torch.float32
    check_calls(pool, twin, ("step", "split", "3frames", "step"), B, T, 3, dtype)


# ---------------------------------------------------------------- 8. CUDA graph
@pytest.mark.gpu
@pytest.mark.parametrize("m,P,B", ((16, 900, 400), (32, 1000, 600), (8, 40, 6)))
@pytest.mark.parametrize("dtype", DTYPES)
def test_graph_replays_any_ids(pq, mods, dtype, m, P, B):
    """One captured half step with CUDA ids replays with new ids and blocks: bit-equal to an eager half pool (native and staged shapes)."""
    mod = mods(100, m)
    graph_pool, eager = pq.StreamPool(mod, P, dtype=dtype), pq.StreamPool(mod, P, dtype=dtype)
    rng = np.random.default_rng(P + B)
    pre = torch.from_numpy(rng.choice(P, P // 3, replace=False).astype(np.int32)).cuda()  # mixed parities first
    xpre = blocks((pre.numel(), 1, 3 * m), 9, dtype)
    graph_pool.step(xpre, pre)
    eager.step(xpre, pre)
    static_x = torch.zeros(B, 1, 2048, dtype=dtype, device="cuda")
    static_ids = torch.arange(B, dtype=torch.int32, device="cuda")
    warm = pq.StreamPool(mod, P, dtype=dtype)  # first launches set the kernels' shared-memory limits: not inside a capture
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        warm.step(static_x, static_ids)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        g_out, g_y = graph_pool.step(static_x, static_ids)
    for k in range(5):
        ids = torch.from_numpy(rng.choice(P, B, replace=False).astype(np.int32)).cuda()
        x = blocks((B, 1, 2048), 50 + k, dtype)
        static_x.copy_(x)
        static_ids.copy_(ids)
        graph.replay()
        out, y = eager.step(x, ids)
        assert torch.equal(g_y, y) and torch.equal(g_out, out) and pools_equal(graph_pool, eager), k


# ---------------------------------------------------------------- 9. C outputs inside guard words
@pytest.mark.gpu
@pytest.mark.parametrize("m", [8, 16, 32])
@pytest.mark.parametrize("dtype", DTYPES)
def test_write_guards(pq, mods, dtype, m):
    """A native C step with a partial last tile, a dead row and mixed parities writes nothing outside y, out and the pools, whose margins
    hold guard words, and equals the op on plain buffers."""
    c = _cabi(pq)
    mod = mods(100, m)
    L = mod.hk.shape[1]
    T = 2048
    B, _ = geometry_shape(mod, "T=2048")
    assert native(mod, B, T)
    P = B + 5
    hk, tab, fl = mod.hk.float().contiguous(), mod._tables, mod._flags
    st = torch.cuda.current_stream().cuda_stream
    margin = 4 * T + 64

    def guarded(n):
        buf = torch.full((n + 2 * margin,), GUARD, dtype=torch.int16, device="cuda")
        return buf, buf[margin:margin + n].view(dtype)

    def intact(buf):
        return bool((buf[:margin] == GUARD).all()) and bool((buf[-margin:] == GUARD).all())

    rng = np.random.default_rng(B)
    ids = torch.from_numpy(rng.choice(P, B, replace=False).astype(np.int32)).cuda()
    ids[B // 2] = -1
    ref = pq.StreamPool(mod, P, dtype=dtype)
    ref.xphase.copy_(torch.from_numpy(rng.integers(0, 4, P).astype(np.int32)))
    ref.sphase.copy_(torch.from_numpy(rng.integers(0, 4, P).astype(np.int32)))
    ref.xpool.copy_(blocks(ref.xpool.shape, 1, torch.float32))
    ref.spool.copy_(blocks(ref.spool.shape, 2, torch.float32))
    fmargin = 4 * L + 64
    xpbuf = torch.full((2 * P * L + 2 * fmargin,), 0x7FC0DEAD, dtype=torch.int32, device="cuda").view(torch.float32)
    spbuf = xpbuf.clone()
    xpool, spool = xpbuf[fmargin:-fmargin], spbuf[fmargin:-fmargin]
    xpool.copy_(ref.xpool.flatten())
    spool.copy_(ref.spool.flatten())
    xph, sph = ref.xphase.clone(), ref.sphase.clone()
    ybuf, y = guarded(B * T)
    obuf, out = guarded(B * T)
    x = blocks((B, 1, T), 4, dtype)
    assert c.pqmf_stream_pool_step_x(x.data_ptr(), y.data_ptr(), out.data_ptr(), hk.data_ptr(), tab.data_ptr(), xpool.data_ptr(), xph.data_ptr(),
                                     spool.data_ptr(), sph.data_ptr(), P, ids.data_ptr(), B, T, m, L, fl, CODE[dtype], st) == 0
    torch.cuda.synchronize()
    assert intact(ybuf) and intact(obuf)
    for buf in (xpbuf, spbuf):
        w = buf.view(torch.int32)
        assert bool((w[:fmargin] == 0x7FC0DEAD).all()) and bool((w[-fmargin:] == 0x7FC0DEAD).all())
    out_r, y_r = ref.step(x, ids)
    assert torch.equal(y.view(B, m, T // m), y_r) and torch.equal(out.view(B, 1, T), out_r)
    assert not y_r[B // 2].any() and not out_r[B // 2].any()
    assert torch.equal(xpool.view(ref.xpool.shape), ref.xpool) and torch.equal(spool.view(ref.spool.shape), ref.spool)
    assert torch.equal(xph, ref.xphase) and torch.equal(sph, ref.sphase)


# ---------------------------------------------------------------- 10. errors
@pytest.mark.gpu
def test_errors(pq, mods):
    mod = mods(100, 16)
    for bad in (torch.float64, torch.int16, "bfloat16"):
        with pytest.raises(ValueError):
            pq.StreamPool(mod, 8, dtype=bad)
    assert pq.StreamPool(mod, 8).dtype == torch.float32
    for dtype, other, name in ((torch.bfloat16, torch.float32, "Float"), (torch.float16, torch.bfloat16, "BFloat16"),
                               (torch.bfloat16, torch.float16, "Half")):
        pool = pq.StreamPool(mod, 16, dtype=dtype)
        assert pool.dtype == dtype
        n0 = pq.launch_count()
        with pytest.raises(RuntimeError, match=name):
            pool.step(torch.zeros(3, 1, 256, dtype=other, device="cuda"), [0, 1, 2])
        with pytest.raises(RuntimeError, match=name):
            pool.forward(torch.zeros(3, 1, 256, dtype=other, device="cuda"), [0, 1, 2])
        with pytest.raises(RuntimeError, match=name):
            pool.inverse(torch.zeros(3, 16, 16, dtype=other, device="cuda"), [0, 1, 2])
        with pytest.raises(RuntimeError, match=name):
            pool.step_groups([(torch.zeros(3, 1, 256, dtype=other, device="cuda"), [0, 1, 2])])
        with pytest.raises(RuntimeError, match=name):
            pool.inverse_groups([(torch.zeros(3, 16, 16, dtype=other, device="cuda"), [0, 1, 2])])
        assert pq.launch_count() == n0
        with pytest.raises(RuntimeError, match="not differentiable"):
            pool.inverse(torch.zeros(3, 16, 16, dtype=dtype, device="cuda", requires_grad=True), [0, 1, 2])
        with pytest.raises(RuntimeError, match="not differentiable"):
            pool.inverse_groups([(torch.zeros(3, 16, 16, dtype=dtype, device="cuda", requires_grad=True), [0, 1, 2])])
        with pytest.raises(RuntimeError, match="ids has 3 entries"):
            pool.step(torch.zeros(4, 1, 256, dtype=dtype, device="cuda"), torch.tensor([0, 1, 2], device="cuda"))
        with pytest.raises(ValueError):
            pool.step(torch.zeros(3, 1, 256, dtype=dtype, device="cuda"), [0, 1, 16])
        with pytest.raises(RuntimeError):
            pool.step(torch.zeros(3, 256, dtype=dtype, device="cuda"), [0, 1, 2])  # wrong rank
        with pytest.raises((RuntimeError, NotImplementedError)):
            pool.step(torch.zeros(3, 1, 256, dtype=dtype), [0, 1, 2])  # CPU block
        assert (pool.xphase == 0).all() and (pool.sphase == 0).all() and not pool.xpool.any() and not pool.spool.any()
    # the float32 calls of the op layer keep their contract; the _x ops refuse a dtype outside the three
    with pytest.raises(RuntimeError):
        torch.ops.pqmf_b200.stream_pool_analysis_x(torch.zeros(3, 1, 256, dtype=torch.float64, device="cuda"), mod.hk, mod._tables,
                                                   pool.xpool, pool.xphase, torch.arange(3, dtype=torch.int32, device="cuda"), torch.float64,
                                                   mod._flags)
    # n_band 1: the identity, dtype still checked
    one = pq.CachedPQMF(100, 16).cuda()
    p1 = pq.StreamPool(one, 4, dtype=torch.bfloat16)
    one.n_band = 1  # as the reference's identity module (pqmf.py:250, :280)
    x = torch.randn(2, 1, 64, device="cuda").bfloat16()
    out, y = p1.step(x, [0, 1])
    assert out is x and y is x and p1.forward(x, [0, 1]) is x and p1.inverse(x, [0, 1]) is x
    with pytest.raises(RuntimeError, match="Float"):
        p1.step(x.float(), [0, 1])


# ---------------------------------------------------------------- 11. C argument checks (no GPU)
def test_cabi_argument_checks_happen_before_any_cuda_call(pq):
    """The three _x entries validate on the host and return PQMF_ERR_ARG (or 0 for no rows) without touching a device."""
    c = _cabi(pq)
    an, sy, st = c.pqmf_stream_pool_analysis_x, c.pqmf_stream_pool_synthesis_x, c.pqmf_stream_pool_step_x
    n6, n9 = [None] * 6, [None] * 9
    for code in (DT_F16, DT_BF16):
        # null pointers
        assert an(*n6, 8, None, 4, 2048, 16, 512, 0, code, None) == ERR_ARG
        assert sy(*n6, 8, None, 4, 128, 16, 512, 0, code, None) == ERR_ARG
        assert st(*n9, 8, None, 4, 2048, 16, 512, 0, code, None) == ERR_ARG
        # P < 1, more rows than streams
        for P, n in ((0, 0), (-1, 1), (3, 4)):
            assert an(*n6, P, None, n, 2048, 16, 512, 0, code, None) == ERR_ARG
            assert sy(*n6, P, None, n, 128, 16, 512, 0, code, None) == ERR_ARG
            assert st(*n9, P, None, n, 2048, 16, 512, 0, code, None) == ERR_ARG
        # T % M != 0, empty blocks
        assert an(*n6, 8, None, 4, 2049, 16, 512, 0, code, None) == ERR_ARG
        assert st(*n9, 8, None, 4, 2049, 16, 512, 0, code, None) == ERR_ARG
        assert an(*n6, 8, None, 4, 0, 16, 512, 0, code, None) == ERR_ARG
        assert sy(*n6, 8, None, 4, 0, 16, 512, 0, code, None) == ERR_ARG
        # no rows: nothing to do
        assert an(*n6, 8, None, 0, 2048, 16, 512, 0, code, None) == 0
        assert sy(*n6, 8, None, 0, 128, 16, 512, 0, code, None) == 0
        assert st(*n9, 8, None, 0, 2048, 16, 512, 0, code, None) == 0
    # an unknown dtype code is an argument error, whatever else the call holds
    for code in (-1, 3, 7):
        assert an(*n6, 8, None, 0, 2048, 16, 512, 0, code, None) == ERR_ARG
        assert sy(*n6, 8, None, 0, 128, 16, 512, 0, code, None) == ERR_ARG
        assert st(*n9, 8, None, 0, 2048, 16, 512, 0, code, None) == ERR_ARG
    # PQMF_DTYPE_F32 is the _f32 entry: its own checks
    assert an(*n6, 8, None, 4, 2048, 16, 512, 0, DT_F32, None) == ERR_ARG
    assert st(*n9, 8, None, 0, 2048, 16, 512, 0, DT_F32, None) == 0
