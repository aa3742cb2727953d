"""The streaming Hankel-4 kernels on every bank and block geometry they serve: lockstep, stream pools and int16 PCM blocks.

The streaming kernels read no fixed geometry: h4_analysis_stream_plan / h4_synthesis_stream_plan (pqmf_b200.cu) derive it per call from
the bank's tap span -- history rows (analysis) or frames (synthesis) in front of every block, the window pad that makes the history whole
plane rows, the region pitch and streams per tile, where the roll starts -- and refuse some banks in one direction only.  The sweep here is
attenuation 50 ... 140 x n_band 8 / 16 / 32.  Each shape checks which kernels really ran (the PCM entries return 0 exactly where the fp32
call runs the streaming Hankel-4 kernels), the float64 streaming oracle on rows of the first, second-to-last and partial last tile, the
plain-fp32 module, and the carried state bit for bit after every block (the roll copies values).  The first test needs no GPU: it pins
the plans, restated in Python, to the table below, so that the sweep cannot go vacuous when trims, tap spans or the plans change."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import pqmf_oracle as O

TOL = 1e-5
ATTENUATIONS = [50, 60, 70, 80, 90, 100, 110, 120, 130, 140]
BANDS = [8, 16, 32]
ERR_UNSUPPORTED = -2
NAN_BITS = 0x7FC0DEAD  # guard word: a quiet NaN no kernel writes
N_SM = 148


# (n_band, attenuation) -> L, first tap jlo, taps kt, split into two tap ranges,
#                          analysis (history rows, pad bytes), synthesis (history frames, pad bytes); None: the plan refuses the bank
def _row(L, jlo, kt, split, a, s):
    return dict(L=L, jlo=jlo, kt=kt, split=split, analysis=a, synthesis=s)


BANK_TABLE = {
    **{(8, a): _row(128, 0, 128, False, (2, 0), (16, 0)) for a in (50, 60, 70)},
    **{(8, a): _row(256, 32, 192, False, (4, 64), (32, 64)) for a in (80, 90, 100)},
    **{(8, a): _row(256, 0, 256, False, (4, 0), (32, 0)) for a in (110, 120, 130)},
    (8, 140): _row(512, 96, 320, False, (7, 64), (56, 64)),  # 52 frames of taps, rounded up to 7 rows (K = 64)
    (16, 50): _row(256, 32, 192, False, None, None),  # n_band 16 streams natively at L = 512 only
    **{(16, a): _row(256, 0, 256, False, None, None) for a in (60, 70)},
    **{(16, a): _row(512, 64, 384, False, (7, 0), (28, 0)) for a in (80, 90, 100)},
    **{(16, a): _row(512, 0, 512, False, (8, 0), (32, 0)) for a in (110, 120, 130)},
    (16, 140): _row(1024, 224, 576, False, None, None),
    (32, 50): _row(512, 64, 384, False, (7, 0), None),  # synthesis history of 14 frames: not whole frame quads
    (32, 60): _row(512, 32, 448, False, (8, 64), (16, 64)),
    (32, 70): _row(512, 0, 512, False, (8, 0), (16, 0)),
    (32, 80): _row(1024, 192, 640, False, (13, 0), None),  # 26 frames
    (32, 90): _row(1024, 160, 704, False, (14, 64), (28, 64)),
    (32, 100): _row(1024, 128, 768, False, (14, 0), (28, 0)),
    (32, 110): _row(1024, 64, 448, True, None, None),  # split banks: two launches, never streamed on the Hankel-4 kernels
    (32, 120): _row(1024, 32, 480, True, None, None),
    (32, 130): _row(1024, 0, 512, True, None, None),
    (32, 140): _row(2048, 448, 576, True, None, None),
}
ALL_BANKS = [(a, m) for m in BANDS for a in ATTENUATIONS]
NATIVE_BANKS = [(a, m) for (a, m) in ALL_BANKS if BANK_TABLE[(m, a)]["analysis"] is not None]
ASYMMETRIC_BANKS = [(a, m) for (a, m) in NATIVE_BANKS if BANK_TABLE[(m, a)]["synthesis"] is None]
# block geometry: the default banks, n_band 8 at attenuation 50 (two history rows: 16 streams per tile at 256 samples) and n_band 32 at
# attenuation 90 (pads in both directions)
GEOMETRY_BANKS = [(100, 8), (100, 16), (100, 32), (50, 8), (90, 32)]


@pytest.fixture(scope="module")
def pq():
    import pqmf_b200

    return pqmf_b200


@pytest.fixture(scope="module")
def bank(pq):
    """CachedPQMF modules by (role, attenuation, n_band, device): the prototype design runs scipy's fmin on the host.  role "mod" and
    "twin" are two identical modules, "fp32" the plain-fp32 one.  Every call returns the module with its streaming state reset."""
    cache = {}

    def get(attenuation, n_band, role="mod", device="cuda"):
        key = (role, attenuation, n_band, device)
        if key not in cache:
            cache[key] = pq.CachedPQMF(attenuation, n_band, fp32=role == "fp32").to(device)
        mod = cache[key]
        mod.reset_stream()
        return mod

    return get


# ---------------------------------------------------------------- the plans, restated
def taps(flags):
    """(jlo, kt) of the bank's Hankel-4 images (PQMF_FLAG_TAPS)"""
    return 32 * ((flags >> 8) & 0xF), 32 * ((flags >> 12) & 0x1F)


def _shape_fits(m, kt, synthesis, pad):
    """h4_shape + h4_shape_fits of a CTA-pair launch"""
    ks = (kt + 64 - m + 15) // 16
    rows = 128 + (32 * ks + (6 * m if synthesis else 0) + pad - 1) // 128
    plane = -(-rows * 128 // 1024) * 1024
    return rows <= 144 and ks * 2 * 96 * 16 + 4 * plane + 128 <= 227 * 1024


def bank_plan(pq, mod):
    """The shape-independent part of both plans: ((history rows, pad bytes) of the analysis, (history frames, pad bytes) of the
    synthesis), None for a direction the plan refuses whatever the shape."""
    lib = pq._lib
    m, L = mod.hk.shape
    flags = mod._flags
    jlo, kt = taps(flags)
    if mod._tables.numel() == 0 or flags & (lib.PQMF_FLAG_NO_SIGN | lib.PQMF_FLAG_FP32):
        return None, None
    if (m, L) == (16, 512):
        family = True
    else:
        family = m in (8, 32) and L in (16 * m, 32 * m, 64 * m)
    if not family or kt == 0 or flags & (lib.PQMF_FLAG_H4_SPLIT | lib.PQMF_FLAG_NO_PAIR | lib.PQMF_FLAG_FOLD):
        return None, None
    hist = -(-(L - jlo) // 64) * 64
    a_pad = 2 * (hist - (L - jlo))
    a = (hist // 64, a_pad) if hist <= L and L % 8 == 0 and _shape_fits(m, kt, False, a_pad) else None
    taps_frames = (jlo + kt) // m
    frames = -(-taps_frames * m // 64) * 64 // m
    s_pad = 2 * m * (frames - taps_frames)
    s = (frames, s_pad) if frames % 4 == 0 and frames <= L // m and _shape_fits(m, kt, True, s_pad) else None
    return a, s


def hist_rows(m, plan, direction):
    """history rows in front of every block"""
    return plan[0] if direction == "analysis" else plan[0] * m // 64


def stream_geom(T, hrows):
    """h4_stream_geom: (pitch, streams per tile)"""
    pitch = (T // 64 + hrows + 3) & ~3
    return pitch, 128 // pitch


def native(mod, plan, direction, B, T):
    """the plan accepts B rows of T samples (F = T / n_band frames) in this direction"""
    m, L = mod.hk.shape
    if plan is None or T % 256 != 0 or T < L:
        return False
    pitch, spt = stream_geom(T, hist_rows(m, plan, direction))
    return pitch <= 128 and spt >= 1 and -(-B // spt) >= 96


def largest_native_block(mod, plan, direction):
    m, L = mod.hk.shape
    return max((T for T in range(256, 16385, 256) if native(mod, plan, direction, 1 << 20, T)), default=None)


def spt_of(mod, plan, direction, T):
    return stream_geom(T, hist_rows(mod.hk.shape[0], plan, direction))[1]


# ---------------------------------------------------------------- 1. bank table (no GPU)
def test_bank_table(pq, bank):
    seen_rows, pads, asymmetric = set(), set(), 0
    for att, m in ALL_BANKS:
        mod = bank(att, m, device="cpu")
        want = BANK_TABLE[(m, att)]
        L = mod.hk.shape[1]
        assert (L, *taps(mod._flags)) == (want["L"], want["jlo"], want["kt"]), (m, att)
        assert bool(mod._flags & pq._lib.PQMF_FLAG_H4_SPLIT) == want["split"], (m, att)
        a, s = bank_plan(pq, mod)
        assert (a, s) == (want["analysis"], want["synthesis"]), (m, att, a, s)
        # largest native block: history rows + block rows fill the 128 rows of one tile; the next 256 samples are refused
        for direction, plan in (("analysis", a), ("synthesis", s)):
            t_max = largest_native_block(mod, plan, direction)
            if plan is None:
                assert t_max is None
                continue
            assert t_max == (128 - hist_rows(m, plan, direction)) // 4 * 256, (m, att, direction)
            assert stream_geom(t_max, hist_rows(m, plan, direction)) == (128, 1)
            assert not native(mod, plan, direction, 1 << 20, t_max + 256)
            pads.add((direction, m == 32, plan[1]))
        if a is not None:
            seen_rows.add(a[0])
            asymmetric += s is None
            if s is not None:
                seen_rows.add(hist_rows(m, s, "synthesis"))
            assert native(mod, a, "analysis", 96 * spt_of(mod, a, "analysis", 2048), 2048)
            assert not native(mod, a, "analysis", 95 * spt_of(mod, a, "analysis", 2048), 2048)
    # what the GPU sweep below must keep covering
    assert {2, 4, 7, 8, 13, 14} <= seen_rows, seen_rows
    assert {(d, n32, p) for d in ("analysis", "synthesis") for n32 in (False, True) for p in (0, 64)} <= pads, pads
    assert asymmetric >= 1 and set(ASYMMETRIC_BANKS) == {(50, 32), (80, 32)}
    assert sorted({BANK_TABLE[(m, a)]["L"] for a, m in ALL_BANKS}) == [128, 256, 512, 1024, 2048]


# ---------------------------------------------------------------- GPU helpers
def _cabi(pq):
    c = pq._lib.cabi
    vp, i, lg, u = ctypes.c_void_p, ctypes.c_int, ctypes.c_long, ctypes.c_uint
    c.pqmf_analysis_stream_pcm16.argtypes = [vp] * 6 + [i, lg, i, i, i, i, i, u, vp]
    c.pqmf_synthesis_stream_pcm16.argtypes = [vp] * 6 + [i, i, lg, i, i, i, u, vp]
    c.pqmf_stream_step_pcm16.argtypes = [vp] * 9 + [i, lg, i, i, i, i, i, i, u, vp]
    c.pqmf_stream_pool_step_f32.argtypes = [vp] * 9 + [i, vp, i, lg, i, i, u, vp]
    for f in (c.pqmf_analysis_stream_pcm16, c.pqmf_synthesis_stream_pcm16, c.pqmf_stream_step_pcm16, c.pqmf_stream_pool_step_f32):
        f.restype = ctypes.c_int
    return c


def route(pq, mod, B, T):
    """(analysis, synthesis, step) return codes of the mono PCM entries on B aligned rows of T samples: 0 exactly where the fp32 call
    with the same rows runs the streaming Hankel-4 kernels, PQMF_ERR_UNSUPPORTED (nothing launched) elsewhere"""
    c = _cabi(pq)
    m, L = mod.hk.shape
    hk, tab, fl = mod.hk.float().contiguous(), mod._tables, mod._flags
    st = torch.cuda.current_stream().cuda_stream
    pcm = torch.zeros(B, T, 1, dtype=torch.int16, device="cuda")
    y = torch.empty(B, m, T // m, device="cuda")
    out = torch.empty(B, T, 1, dtype=torch.int16, device="cuda")
    xs, ss = torch.zeros(2, B, L, device="cuda"), torch.zeros(2, B, L, device="cuda")
    ra = c.pqmf_analysis_stream_pcm16(pcm.data_ptr(), y.data_ptr(), hk.data_ptr(), tab.data_ptr(), xs[0].data_ptr(), xs[1].data_ptr(),
                                      B, T, 1, 0, m, L, 0, fl, st)
    rs = c.pqmf_synthesis_stream_pcm16(y.data_ptr(), out.data_ptr(), hk.data_ptr(), tab.data_ptr(), ss[0].data_ptr(), ss[1].data_ptr(),
                                       B, 1, T // m, m, L, 0, fl, st)
    rstep = c.pqmf_stream_step_pcm16(pcm.data_ptr(), y.data_ptr(), out.data_ptr(), hk.data_ptr(), tab.data_ptr(), xs[0].data_ptr(),
                                     xs[1].data_ptr(), ss[0].data_ptr(), ss[1].data_ptr(), B, T, 1, 0, m, L, 0, 0, fl, st)
    torch.cuda.synchronize()
    return ra, rs, rstep


def expected_route(pq, mod, B, T):
    a, s = bank_plan(pq, mod)
    na, ns = native(mod, a, "analysis", B, T), native(mod, s, "synthesis", B, T)
    rc = lambda ok: 0 if ok else ERR_UNSUPPORTED  # noqa: E731
    return rc(na), rc(ns), rc(na and ns)


def check_route(pq, mod, B, T):
    want = expected_route(pq, mod, B, T)
    assert route(pq, mod, B, T) == want, (mod.n_band, B, T, want)
    return want


def blocks(B, t, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (0.5 * torch.randn(B, 1, t, device="cuda", generator=g)).clamp_(-1, 1)


def call_rows(pq, mod, T, n_tiles=101):
    """(B, spt): B streams of T samples on n_tiles tiles of the analysis plan (spt streams each), the last one partial (one live stream);
    banks the plan refuses get the same sizes as if three streams shared a tile"""
    a, _ = bank_plan(pq, mod)
    spt = max(spt_of(mod, a, "analysis", T), 1) if a is not None else 3
    return (spt * (n_tiles - 1) + 1 if spt > 1 else n_tiles), spt


def sample_rows(B, spt, extra=()):
    """the first rows, a middle row, every row of the second-to-last and the (partial) last tile: at least 8"""
    n_tiles = -(-B // spt)
    rows = {0, 1, B // 2, *extra} | set(range(max(0, (n_tiles - 2) * spt), B))
    r = 2
    while len(rows) < 8:
        rows.add(r)
        r += 1
    return sorted(x for x in rows if x < B)


def run_lockstep(bank, att, m, B, T, rows, seed, plan=("step", "split", "3frames", "step", "step"), fp32_twin=True):
    """Blocks of B streams through process_stream / forward_stream + inverse_stream (a 3-frame block in the middle: the native kernels run
    at both frame parities).  After every block: both state halves bit-equal to the last L samples / K frames of (history ++ block), the
    plain-fp32 module within 3e-6 / 8e-6, and `rows` against the float64 streaming oracle within TOL / 2.  Returns the module."""
    mod = bank(att, m)
    ref = bank(att, m, "fp32") if fp32_twin else None
    L = mod.hk.shape[1]
    K = L // m
    hk = mod.hk.cpu().double().numpy()
    st = O.StreamState(len(rows), m, L)
    ridx = torch.tensor(rows, device="cuda")
    xs_prev = torch.zeros(B, L, device="cuda")
    ss_prev = torch.zeros(B, m, K, device="cuda")
    for k, kind in enumerate(plan):
        x = blocks(B, 3 * m if kind == "3frames" else T, seed + k)
        if kind == "split":
            y = mod.forward_stream(x)
            out = mod.inverse_stream(y)
        else:
            out, y = mod.process_stream(x)
        xs_new = torch.cat([xs_prev, x[:, 0]], -1)[:, -L:]
        ss_new = torch.cat([ss_prev, y], -1)[..., -K:]
        assert torch.equal(mod._x_state[mod._x_slot], xs_new), ("analysis state", k)
        assert torch.equal(mod._s_state[mod._s_slot].view(B, m, K), ss_new), ("synthesis state", k)
        xs_prev, ss_prev = xs_new, ss_new
        if ref is not None:  # each direction on the same input: the synthesis gain (n_band) would amplify analysis differences
            y_p = ref.forward_stream(x)
            out_p = ref.inverse_stream(y)
            assert (y - y_p).abs().max().item() <= 3e-6 and (out - out_p).abs().max().item() <= 8e-6, k
        y64 = O.stream_analysis(x[ridx, 0].cpu().double().numpy(), hk, st)
        o64 = O.stream_synthesis(y[ridx].cpu().double().numpy(), hk, st)
        ea = np.abs(y[ridx].cpu().numpy() - y64).max(axis=(1, 2))
        es = np.abs(out[ridx, 0].cpu().numpy() - o64).max(axis=1)
        assert ea.max() <= TOL / 2, ("analysis", k, rows[int(ea.argmax())], float(ea.max()))
        assert es.max() <= TOL / 2, ("synthesis", k, rows[int(es.argmax())], float(es.max()))
    return mod


# ---------------------------------------------------------------- 3. every bank, lockstep
@pytest.mark.gpu
@pytest.mark.parametrize("att,m", ALL_BANKS)
def test_every_bank_lockstep(pq, bank, att, m):
    mod = bank(att, m)
    a, s = bank_plan(pq, mod)
    T = 2048
    B, spt = call_rows(pq, mod, T)
    rc = check_route(pq, mod, B, T)
    assert rc[0] == (0 if a is not None else ERR_UNSUPPORTED) and rc[1] == (0 if s is not None else ERR_UNSUPPORTED)
    for plan, direction in ((a, "analysis"), (s, "synthesis")):
        if plan is not None:  # odd tile count, partial last tile in both directions
            n = spt_of(mod, plan, direction, T)
            assert -(-B // n) % 2 == 1 and B % n != 0, (direction, n)
    run_lockstep(bank, att, m, B, T, sample_rows(B, spt), seed=att * 100 + m)
    # few streams: the fold kernels (n_band 16 / L 512) or the direct form, every row against the oracle
    assert check_route(pq, mod, 5, T) == (ERR_UNSUPPORTED,) * 3
    run_lockstep(bank, att, m, 5, T, list(range(5)), seed=att * 100 + m + 50, plan=("step", "3frames", "split"))


# ---------------------------------------------------------------- 4. every native bank: pools and PCM
def _pool_reference(mod, x, ids, xpool, spool, xphase, sphase, B):
    """What stream_step gives each listed stream on its own state, grouped by (analysis, synthesis) parity; each group padded with
    zero streams to the call's B rows, so it runs on the same kernels as the pool call."""
    n, T = x.shape[0], x.shape[-1]
    m = mod.n_band
    y = torch.empty(n, m, T // m, device="cuda")
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

            def padded(t):
                return torch.cat([t, t.new_zeros((B - g,) + tuple(t.shape[1:]))])

            xs_in, ss_in = padded(xpool[xh[sel], idl[sel]]), padded(spool[sh[sel], idl[sel]].reshape(g, -1))
            xs_out, ss_out = torch.empty_like(xs_in), torch.empty_like(ss_in)
            o, yy = torch.ops.pqmf_b200.stream_step(padded(x[sel]), mod.hk.float(), mod._tables, xs_in, xs_out, ss_in, ss_out, a, b, mod._flags)
            y[sel], out[sel], xnew[sel], snew[sel] = yy[:g], o[:g], xs_out[:g], ss_out[:g]
    return out, y, xnew, snew


def pool_step_checked(pool, mod, x, ids, dead, B):
    """pool.step with CUDA ids (row `dead` carries an id outside the pool): live rows bit-equal to the lockstep entry on each stream's own
    state and parity, the dead row zeros, streams not listed untouched in both halves and both phase words"""
    P = pool.capacity
    live = torch.ones(ids.numel(), dtype=torch.bool, device="cuda")
    live[dead] = False
    before = [t.clone() for t in (pool.xpool, pool.spool, pool.xphase, pool.sphase)]
    out_r, y_r, xnew_r, snew_r = _pool_reference(mod, x[live], ids[live], *before, B)
    out, y = pool.step(x, ids)
    assert torch.equal(y[live], y_r) and torch.equal(out[live], out_r)
    assert not y[dead].any() and not out[dead].any()
    idl = ids[live].long()
    assert torch.equal(pool.xpool[pool.xphase[idl].long() & 1, idl], xnew_r)
    assert torch.equal(pool.spool[pool.sphase[idl].long() & 1, idl].reshape(idl.numel(), -1), snew_r)
    rest = torch.ones(P, dtype=torch.bool, device="cuda")
    rest[idl] = False
    assert torch.equal(pool.xpool[:, rest], before[0][:, rest]) and torch.equal(pool.spool[:, rest], before[1][:, rest])
    assert torch.equal(pool.xphase[rest], before[2][rest]) and torch.equal(pool.sphase[rest], before[3][rest])
    return out, y


@pytest.mark.gpu
@pytest.mark.parametrize("att,m", NATIVE_BANKS)
def test_every_native_bank_pool(pq, bank, att, m):
    """297 tiles (odd; CTAs run two or three of them, so a drain and the next tile's convert carry different streams' parities), streams
    at mixed frame parities, a seeded permutation of ids over a larger pool, one dead row."""
    mod = bank(att, m)
    T = 2048
    B, _ = call_rows(pq, mod, T, n_tiles=2 * N_SM + 1)
    assert check_route(pq, mod, B, T)[0] == 0
    P = B + 37
    pool = pq.StreamPool(mod, P)
    rng = np.random.default_rng(att * 10 + m)
    pre_step(pool, rng, m)
    for k in range(3):
        ids = torch.from_numpy(rng.choice(P, B, replace=False).astype(np.int32)).cuda()
        dead = int(rng.integers(B))
        ids[dead] = P + 3
        pool_step_checked(pool, mod, blocks(B, T, 10 + k), ids, dead, B)


def pre_step(pool, rng, m):
    """a 3-frame block (direct form) on a random third of the pool: neighbouring tiles of the next calls carry different signs"""
    P = pool.capacity
    pre = torch.from_numpy(rng.choice(P, P // 3, replace=False).astype(np.int32)).cuda()
    x = blocks(pre.numel(), 3 * m, 1)
    out, y = pool.step(x, pre)
    assert ((pool.xphase >> 1) & 1).sum().item() == pre.numel()
    return pre, x, out, y


def widen(pcm, downmix):
    """[S, T, C] int16 -> [S, C', T] float32, the kernels' arithmetic (a tensor divisor: torch divides by a host scalar via its reciprocal)"""
    f = pcm.to(torch.float32) * (1.0 / 32768.0)
    if not downmix:
        return f.permute(0, 2, 1).contiguous()
    acc = f[..., 0].clone()
    for c in range(1, f.shape[-1]):
        acc += f[..., c]
    return (acc / torch.tensor(float(f.shape[-1]), device=acc.device)).unsqueeze(1)


def quantise(v):
    """[S, C, T] float32 -> [S, T, C] int16"""
    return (v * 32768.0).round().clamp(-32768, 32767).to(torch.int16).permute(0, 2, 1).contiguous()


def pcm_blocks(shape, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (8000.0 * torch.randn(shape, device="cuda", generator=g)).round().clamp(-32768, 32767).to(torch.int16)


@pytest.mark.gpu
@pytest.mark.parametrize("att,m", NATIVE_BANKS)
def test_every_native_bank_pcm(pq, bank, att, m):
    """process_stream_pcm16 / forward_stream_pcm16, mono and stereo down-mix: bit-equal to the fp32 twin on the widened block plus the
    quantisation, the same state.  On the asymmetric banks the PCM analysis is native and the PCM step is staged."""
    mod, twin = bank(att, m), bank(att, m, "twin")
    T = 2048
    B, _ = call_rows(pq, mod, T)
    ra, rs, rstep = check_route(pq, mod, B, T)
    assert ra == 0 and (rs, rstep) == ((ERR_UNSUPPORTED,) * 2 if (att, m) in ASYMMETRIC_BANKS else (0, 0))
    plan = [("step", 1, False), ("forward", 2, True), ("step", 2, True), ("3frames", 1, False), ("forward", 1, False), ("step", 1, False)]
    for k, (kind, C, downmix) in enumerate(plan):
        pcm = pcm_blocks((B, 3 * m if kind == "3frames" else T, C), 1000 * m + att + k)
        xw = widen(pcm, downmix)
        if kind == "forward":
            y = mod.forward_stream_pcm16(pcm, downmix)
            y_r = twin.forward_stream(xw)
            assert torch.equal(y, y_r), (k, kind)
            out, out_r = mod.inverse_stream(y), twin.inverse_stream(y_r)
            assert torch.equal(out, out_r), (k, kind)
        else:
            out, y = mod.process_stream_pcm16(pcm, downmix)
            out_r, y_r = twin.process_stream(xw)
            assert torch.equal(y, y_r) and torch.equal(out, quantise(out_r)), (k, kind)
        assert torch.equal(mod._x_state, twin._x_state) and torch.equal(mod._s_state, twin._s_state), (k, kind)
        assert (mod._x_slot, mod._s_slot, mod._frames_in, mod._frames_out) == (twin._x_slot, twin._s_slot, twin._frames_in, twin._frames_out)


# ---------------------------------------------------------------- 5. block geometry
GEOMETRY_CASES = ["T=L", "T=2048", "T=max", "T=max+256", "tiles=95", "tiles=96", "tiles=97"]


def geometry_shape(pq, mod, case):
    """(B, T) of a case: T = max(L, 256) (every block group rolls where T == L), the config-3 block, the largest native block (one stream
    per tile, pitch 128) and the next one (refused), and 95 / 96 / 97 tiles at 2048 samples around the threshold; partial last tiles"""
    a, s = bank_plan(pq, mod)
    L = mod.hk.shape[1]
    t_max = largest_native_block(mod, a, "analysis")
    assert t_max == largest_native_block(mod, s, "synthesis")  # the geometry banks have as many history rows in both directions
    T = {"T=L": max(L, 256), "T=max": t_max, "T=max+256": t_max + 256}.get(case, 2048)
    spt = spt_of(mod, a, "analysis", T) if case != "T=max+256" else 1
    n_tiles = int(case.split("=")[1]) if case.startswith("tiles") else 101
    B = spt * (n_tiles - 1) + 1 if spt > 1 else n_tiles
    return B, T, spt


@pytest.mark.gpu
@pytest.mark.parametrize("case", GEOMETRY_CASES)
@pytest.mark.parametrize("att,m", GEOMETRY_BANKS)
def test_block_geometry(pq, bank, att, m, case):
    mod = bank(att, m)
    B, T, spt = geometry_shape(pq, mod, case)
    rc = check_route(pq, mod, B, T)
    assert rc == ((ERR_UNSUPPORTED,) * 3 if case in ("T=max+256", "tiles=95") else (0, 0, 0)), (case, B, T)
    if case == "T=max":
        assert spt == 1
    run_lockstep(bank, att, m, B, T, sample_rows(B, spt), seed=att + m + T, plan=("step", "3frames", "split", "step"))


def _guarded(n, margin):
    """a [margin | n | margin] float32 buffer of guard words; returns (buffer, the inner n floats)"""
    buf = torch.full((n + 2 * margin,), NAN_BITS, dtype=torch.int32, device="cuda").view(torch.float32)
    return buf, buf[margin:margin + n]


def _margins_intact(buf, margin):
    w = buf.view(torch.int32)
    return bool((w[:margin] == NAN_BITS).all()) and bool((w[-margin:] == NAN_BITS).all())


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["T=L", "T=2048"])
@pytest.mark.parametrize("att,m", GEOMETRY_BANKS)
def test_write_guards(pq, bank, att, m, case):
    """y, out, state_out and both pools inside buffers whose margins (a tile's rows and more on each side) hold guard words: the C entries
    of the partial last tile and the padding tile of the CTA pair write nothing outside their buffers, and the values equal the torch
    ops' on plain buffers."""
    c = _cabi(pq)
    lib = pq._lib.cabi
    mod = bank(att, m)
    B, T, spt = geometry_shape(pq, mod, case)
    assert check_route(pq, mod, B, T) == (0, 0, 0) and B % spt != 0 and -(-B // spt) % 2 == 1
    L = mod.hk.shape[1]
    F, K = T // m, L // m
    hk, tab, fl = mod.hk.float().contiguous(), mod._tables, mod._flags
    st = torch.cuda.current_stream().cuda_stream
    x = blocks(B, T, 7)
    xs_in = blocks(B, L, 8)[:, 0].contiguous()
    ss_in = blocks(B, L, 9)[:, 0].contiguous()
    # lockstep, both directions
    my = spt * T + 64
    ybuf, y = _guarded(B * T, my)
    xobuf, xs_out = _guarded(B * L, spt * L + 64)
    assert lib.pqmf_analysis_stream_f32(x.data_ptr(), y.data_ptr(), hk.data_ptr(), tab.data_ptr(), xs_in.data_ptr(), xs_out.data_ptr(), B, T, m,
                                        L, 1, fl, st) == 0
    obuf, out = _guarded(B * T, my)
    sobuf, ss_out = _guarded(B * L, spt * L + 64)
    y_s = blocks(B, T, 10).view(B, m, F)
    assert lib.pqmf_synthesis_stream_f32(y_s.data_ptr(), out.data_ptr(), hk.data_ptr(), tab.data_ptr(), ss_in.data_ptr(), ss_out.data_ptr(), B, F,
                                         m, L, 1, fl, st) == 0
    torch.cuda.synchronize()
    for buf, mg in ((ybuf, my), (xobuf, spt * L + 64), (obuf, my), (sobuf, spt * L + 64)):
        assert _margins_intact(buf, mg)
    x_o, s_o = torch.empty(B, L, device="cuda"), torch.empty(B, L, device="cuda")
    assert torch.equal(y.view(B, m, F), torch.ops.pqmf_b200.analysis_stream(x, hk, tab, xs_in, x_o, 1, fl)) and torch.equal(xs_out.view(B, L), x_o)
    assert torch.equal(out.view(B, 1, T), torch.ops.pqmf_b200.synthesis_stream(y_s, hk, tab, ss_in, s_o, 1, fl)) and torch.equal(ss_out.view(B, L), s_o)
    # a pool step: pools, outputs guarded; one dead row; mixed parities
    P = B + 5
    rng = np.random.default_rng(B)
    ids = torch.from_numpy(rng.choice(P, B, replace=False).astype(np.int32)).cuda()
    ids[B // 2] = -1
    xphase = torch.from_numpy(rng.integers(0, 4, P).astype(np.int32)).cuda()
    sphase = torch.from_numpy(rng.integers(0, 4, P).astype(np.int32)).cuda()
    mp = spt * L + 64
    xpbuf, xpool = _guarded(2 * P * L, mp)
    spbuf, spool = _guarded(2 * P * L, mp)
    xpool.copy_(blocks(2 * P, L, 11).flatten())
    spool.copy_(blocks(2 * P, L, 12).flatten())
    pool_ref = pq.StreamPool(mod, P)
    pool_ref.xpool.copy_(xpool.view(2, P, L))
    pool_ref.spool.copy_(spool.view(pool_ref.spool.shape))
    pool_ref.xphase.copy_(xphase)
    pool_ref.sphase.copy_(sphase)
    ybuf, y = _guarded(B * T, my)
    obuf, out = _guarded(B * T, my)
    assert c.pqmf_stream_pool_step_f32(x.data_ptr(), y.data_ptr(), out.data_ptr(), hk.data_ptr(), tab.data_ptr(), xpool.data_ptr(), xphase.data_ptr(),
                                       spool.data_ptr(), sphase.data_ptr(), P, ids.data_ptr(), B, T, m, L, fl, st) == 0
    torch.cuda.synchronize()
    for buf, mg in ((ybuf, my), (obuf, my), (xpbuf, mp), (spbuf, mp)):
        assert _margins_intact(buf, mg)
    out_r, y_r = pool_ref.step(x, ids)
    assert torch.equal(y.view(B, m, F), y_r) and torch.equal(out.view(B, 1, T), out_r)
    assert torch.equal(xpool.view(2, P, L), pool_ref.xpool) and torch.equal(spool.view(pool_ref.spool.shape), pool_ref.spool)
    assert torch.equal(xphase, pool_ref.xphase) and torch.equal(sphase, pool_ref.sphase)


# ---------------------------------------------------------------- 6. steady state of the persistent loop
# n_band 8: 4096 streams x 2048 samples = 1366 tiles of 3; n_band 32: 2960 streams = 1480 tiles of 2, 10 per CTA on 148 SMs.  The oracle
# rows are those of the tiles every CTA c visits on its 1st, 2nd, ... and last iteration, and of the partial last tile.
STEADY = {8: 4096, 32: 2960}


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["lockstep", "pool"])
@pytest.mark.parametrize("m", [8, 32])
def test_steady_state(pq, bank, m, mode):
    B, T = STEADY[m], 2048
    mod = bank(100, m)
    a, _ = bank_plan(pq, mod)
    spt = spt_of(mod, a, "analysis", T)
    n_tiles = -(-B // spt)
    assert n_tiles >= 9 * N_SM and check_route(pq, mod, B, T) == (0, 0, 0)
    rows = sorted({spt * (N_SM * k + c) for k in range(n_tiles // N_SM + 1) for c in (0, 1, 77, N_SM - 1) if spt * (N_SM * k + c) < B}
                  | set(range((n_tiles - 1) * spt, B)))
    if mode == "lockstep":
        run_lockstep(bank, 100, m, B, T, rows, seed=m, plan=("step", "split", "step"), fp32_twin=False)
        return
    # a pool of B + 40 streams at mixed parities, a new permutation every block and one dead row; every row bit-equal to the lockstep
    # entry, and sampled streams -- placed on the oracle rows -- followed through the oracle from their first block
    P = B + 40
    pool = pq.StreamPool(mod, P)
    hk = mod.hk.cpu().double().numpy()
    L = mod.hk.shape[1]
    rng = np.random.default_rng(m)
    sampled = rng.choice(P, len(rows), replace=False)
    oracle = {int(i): O.StreamState(1, m, L) for i in sampled}

    def follow(ids, x, y, out, at):
        for r in at:
            st = oracle[int(ids[r])]
            y64 = O.stream_analysis(x[r:r + 1, 0].cpu().double().numpy(), hk, st)
            o64 = O.stream_synthesis(y[r:r + 1].cpu().double().numpy(), hk, st)
            assert np.abs(y[r:r + 1].cpu().numpy() - y64).max() <= TOL / 2, (r, int(ids[r]))
            assert np.abs(out[r:r + 1, 0].cpu().numpy() - o64).max() <= TOL / 2, (r, int(ids[r]))

    pre, xp, outp, yp = pre_step(pool, rng, m)
    pre = pre.cpu().numpy()
    follow(pre, xp, yp, outp, [r for r in range(len(pre)) if int(pre[r]) in oracle])
    spare = [r for r in range(B) if r not in set(rows)]
    for k in range(3):
        ids = np.empty(B, np.int64)
        ids[rows] = rng.permutation(sampled)
        ids[spare] = rng.permutation(np.setdiff1d(np.arange(P), sampled))[:len(spare)]
        dead = int(rng.choice(spare))
        ids[dead] = P + 3
        x = blocks(B, T, 20 + k)
        out, y = pool_step_checked(pool, mod, x, torch.from_numpy(ids.astype(np.int32)).cuda(), dead, B)
        follow(ids, x, y, out, rows)
