"""The n_band-16 kernels for small calls and few streams -- fold + modulation (f16_analysis_kernel / f16_synthesis_kernel, fast16*.cuh)
and Hankel-16 (h16_analysis_kernel / h16_synthesis_kernel, hankel16.cuh) -- in the steady state of their persistent loops and on every
n_band-16 bank they serve, offline and streaming.

All four are persistent kernels: a CTA walks tiles first, first + grid, ... with double-buffered windows / planes / accumulators and
mbarrier phases that first wrap on a CTA's third tile.  Real callers get there: lockstep streaming with blocks that are not a multiple of
256 samples (the 48 kHz sizes 480, 960, ...), few streams with long blocks, offline buffers the Hankel-4 kernels refuse only for their
alignment, and exact=True on any of them.  The key check needs no tolerance: a tile's output depends only on its own window (and the
carried history), not on which CTA runs it at which iteration, so every row of a steady-state launch must be BIT-EQUAL to the same row
computed by a call small enough that each CTA takes at most one tile (same kernel instantiation: same flags, same F, same delay).  The
float64 oracle then checks the kernels themselves on excerpts placed on the tiles CTA 0, a middle CTA and the last CTA run on their 1st,
2nd, 3rd and last iteration.  Every GPU case first asserts which family ran and how many tiles each CTA takes.  The first test needs no
GPU: it pins the banks' tap spans and the instantiations they select."""
import numpy as np
import pytest
import torch

from oracle import pqmf_oracle as O

TOL = 1e-5
ATTENUATIONS = [50, 60, 70, 80, 90, 100, 110, 120, 130, 140]
FOLD_RESIDUAL_LIMIT = 1e-6  # pqmf.py: a bank above it is marked PQMF_FLAG_NO_FOLD

# attenuation -> L, first tap, taps (PQMF_FLAG_TAPS), fold <QLO, QN>, Hankel-16 <JLO, KT>, fold residual |hk - g (x) C| observed
# (float64 of the fp32 bank; printed per bank here for the first time).  L != 512: none of these kernels exist for the bank.
N16_TABLE = {
    50: (256, 32, 192, None, None, 0.0),
    60: (256, 0, 256, None, None, 0.0),
    70: (256, 0, 256, None, None, 0.0),
    80: (512, 64, 384, (2, 12), (64, 384), 1.6446e-07),
    90: (512, 64, 384, (2, 12), (64, 384), 1.6588e-07),
    100: (512, 64, 384, (2, 12), (64, 384), 1.6634e-07),
    110: (512, 0, 512, (0, 16), (0, 512), 1.6648e-07),
    120: (512, 0, 512, (0, 16), (0, 512), 1.6639e-07),
    130: (512, 0, 512, (0, 16), (0, 512), 1.6717e-07),
    140: (1024, 224, 576, None, None, 0.0),
}
FAMILY_BANKS = [a for a in ATTENUATIONS if N16_TABLE[a][3] is not None]
OTHER_BANKS = [a for a in ATTENUATIONS if N16_TABLE[a][3] is None]

# shapes of the GPU cases below (the table test checks what they cover)
STEADY_ROWS, STEADY_T = 1499, 3 * 2048 - 64  # offline: F = 380, partial last analysis tile, synthesis J = 7
BANK_ROWS = 467                              # every bank: 2-3 tiles per CTA at the same T
LONG_SHAPES = [(64, 1 << 19), (64, (1 << 19) - 3 * 16), (2, 1 << 21)]
STREAM_PLAN = [480, 480, 48, 960, 480, 480]  # 48 kHz blocks; 3 frames (odd parity) and 960 in the middle; 480 < L and F = 30 < K
STREAMS = 4096
EDGE_FRAMES = [1, 2, 3, 127, 128, 129, 160, 161, 224, 225]  # F = 1: a 16-sample signal
EDGE_BLOCKS = [496, 16, 48, 496, 16]                          # T < L at odd frame counts


@pytest.fixture(scope="module")
def pq():
    import pqmf_b200

    return pqmf_b200


@pytest.fixture(scope="module")
def bank(pq):
    """modules by (attenuation, role, class, device): the prototype design runs scipy's fmin on the host.  role "mod" is the default
    module, "twin" a second one like it, "exact" the exact=True one, "fp32" the plain-fp32 twin.  Every call returns the module with its streaming state reset."""
    cache = {}

    def get(attenuation, role="mod", cls="CachedPQMF", device="cuda"):
        key = (attenuation, role, cls, device)
        if key not in cache:
            cache[key] = getattr(pq, cls)(attenuation, 16, exact=role == "exact", fp32=role == "fp32").to(device)
        mod = cache[key]
        if cls == "CachedPQMF":
            mod.reset_stream()
        return mod

    return get


# ---------------------------------------------------------------- the launchers, restated
def taps(flags):
    """(jlo, kt) of the bank's tap span (PQMF_FLAG_TAPS)"""
    return 32 * ((flags >> 8) & 0xF), 32 * ((flags >> 12) & 0x1F)


def instantiations(mod):
    """(fold <QLO, QN>, Hankel-16 <JLO, KT>) the bank's taps select (fast16_taps_from_flags, exact_tc_*); (None, None) where the bank is
    not n_band 16 / L 512 and none of these kernels run"""
    if tuple(mod.hk.shape) != (16, 512):
        return None, None
    trimmed = taps(mod._flags) == (64, 384)
    return ((2, 12), (64, 384)) if trimmed else ((0, 16), (0, 512))


def fold_j(F):
    """FIR outputs per thread of the fold synthesis: J = 4 for streaming-sized blocks (F <= 160), else 7 (fast16_synthesis)"""
    return 4 if F <= 160 else 7


def h16_ctas_per_sm(kt, synthesis, smem_per_sm):
    """h16_launch_*: as many CTAs per SM as the shared memory holds, at most 4 (H16*Smem<KT>::BYTES + 1 KiB reserved each)"""
    ks = kt // 16
    rows = 128 + ks
    plane = -(-rows * 32 // 1024) * 1024
    nbytes = kt * 64 + 4 * plane + (0 if synthesis else 2 * 16 * rows * 4) + 128
    return max(1, min(4, smem_per_sm // (nbytes + 1024)))


KINDS = {"fold": ("fold_a", "fold_s"), "h16": ("h16_a", "h16_s")}


def launch(kind, F, flags):
    """(tiles per row, CTAs of a full grid, frames per tile) of one family and direction for rows of F frames; a launch of B rows runs
    min(CTAs, B x tiles per row) CTAs"""
    p = torch.cuda.get_device_properties(torch.cuda.current_device())
    sm, smem = p.multi_processor_count, p.shared_memory_per_multiprocessor
    kt = 384 if taps(flags) == (64, 384) else 512
    if kind == "fold_a":
        return -(-F // 128), 4 * sm, 128
    if kind == "fold_s":
        ni = 16 * fold_j(F)  # output rows of 32 samples (two frames) per tile
        return -(-(-(-F // 2)) // ni), 2 * sm, 2 * ni
    return -(-F // 128), h16_ctas_per_sm(kt, kind == "h16_s", smem) * sm, 128


def tiles_per_cta(kind, B, F, flags):
    tpr, ctas, _ = launch(kind, F, flags)
    return B * tpr / min(ctas, B * tpr)


def family_flags(pq, flags, family):
    """flags that force one family: FOLD keeps the Hankel-4 kernels off, NO_FOLD (or EXACT) sends the fold path to Hankel-16; "direct" is
    the plain-fp32 twin's route (the register-tiled direct form)"""
    lib = pq._lib
    if family == "fold":
        return (flags & ~(lib.PQMF_FLAG_EXACT | lib.PQMF_FLAG_NO_FOLD)) | lib.PQMF_FLAG_FOLD
    if family == "h16":
        return flags | lib.PQMF_FLAG_FOLD | lib.PQMF_FLAG_NO_FOLD
    return flags | lib.PQMF_FLAG_FP32


def analysis(mod, x, flags):
    return torch.ops.pqmf_b200.analysis(x, mod.hk.float(), mod._tables, x.shape[-1] // 16, flags)


def synthesis(mod, s, delay, flags):
    return torch.ops.pqmf_b200.synthesis(s, mod.hk.float(), mod._tables, delay, flags)


def signal(shape, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (0.5 * torch.randn(shape, device="cuda", generator=g)).clamp_(-1, 1)


def at_offset(t, nbytes):
    """a copy of t that starts nbytes past a 512-byte boundary (the caching allocator's alignment): a contiguous view, which
    .contiguous() does not copy"""
    buf = torch.empty(t.numel() + nbytes // 4 + 64, device=t.device)
    assert buf.data_ptr() % 512 == 0
    v = buf[nbytes // 4:nbytes // 4 + t.numel()].view(t.shape)
    v.copy_(t)
    return v


def one_tile_per_cta(fn, t, kind, F, flags):
    """fn over row chunks of t small enough that each CTA takes at most one tile (fresh aligned copies)"""
    tpr, ctas, _ = launch(kind, F, flags)
    rows = ctas // tpr
    assert rows >= 1, (kind, F, "a row alone is more tiles than the grid")
    return torch.cat([fn(t[i:i + rows].clone()) for i in range(0, t.shape[0], rows)])


def assert_family(got, calls, family):
    """got is bit-equal to calls[family] and differs in bits from every other family's result on the same input"""
    assert torch.equal(got, calls[family]), f"not the {family} result"
    for other, v in calls.items():
        if other != family:
            assert not torch.equal(got, v), f"{family} result bit-equal to the {other} result"


def sampled_tiles(n_tiles, grid):
    """the tiles CTA 0, a middle CTA and the last CTA run on their 1st, 2nd, 3rd and last iteration (tile = it * grid + cta)"""
    out = set()
    for cta in (0, grid // 2, grid - 1):
        last = (n_tiles - 1 - cta) // grid
        for it in {0, 1, 2, last}:
            if 0 <= it * grid + cta < n_tiles:
                out.add(it * grid + cta)
    return sorted(out)


def oracle_excerpts(kind, B, F, flags):
    """(row, first frame, end frame) of the sampled tiles of one launch (tile = b * tpr + c)"""
    tpr, ctas, span = launch(kind, F, flags)
    return [(t // tpr, (t % tpr) * span, min(F, (t % tpr + 1) * span)) for t in sampled_tiles(B * tpr, min(ctas, B * tpr))]


def check_oracle_analysis(x, y, hk, excerpts):
    """offline sub-bands of the excerpts against the float64 oracle on the cropped input they depend on: one filter length of halo on
    each side, cut at an even frame (the sign mask follows the global frame parity) or at the row's ends"""
    halo, F = 32, y.shape[-1]
    for b, lo, hi in excerpts:
        f0, f1 = max(0, lo - halo) & ~1, min(F, hi + halo)
        y64 = O.analysis(x[b, 0, f0 * 16:f1 * 16].cpu().double().numpy()[None], hk)[0]
        err = np.abs(y[b, :, lo:hi].cpu().double().numpy() - y64[:, lo - f0:hi - f0]).max()
        assert err <= TOL / 2, ("analysis", b, lo, hi, float(err))


def check_oracle_synthesis(s, out, hk, delay, excerpts):
    halo, F = 32, s.shape[-1]
    for b, lo, hi in excerpts:
        f0, f1 = max(0, lo - halo) & ~1, min(F, hi + halo)
        o64 = O.synthesis(s[b, :, f0:f1].cpu().double().numpy()[None], hk, delay_frames=delay)[0]
        a = (lo - f0) * 16
        err = np.abs(out[b, 0, lo * 16:hi * 16].cpu().double().numpy() - o64[a:a + (hi - lo) * 16]).max()
        assert err <= TOL / 2, ("synthesis", b, lo, hi, delay, float(err))


def offline_case(pq, mod, x, delay, family, flags=None, s_offset=4, min_tiles=0.0, reference=True):
    """Analysis of x, then synthesis of those sub-bands placed `s_offset` bytes past a 16-byte boundary: through the module (flags None:
    the production route) or the ops with `flags`.  Checks, in order: one launch per direction, the family that ran (bit-equal to the
    forced call, different bits from the other families on the first rows), at least `min_tiles` tiles per CTA, every row bit-equal to
    the one-tile-per-CTA reference, oracle excerpts on the sampled tiles.  Returns (y, out)."""
    B, T = x.shape[0], x.shape[-1]
    F = T // 16
    fl = mod._flags if flags is None else flags
    forced = {f: family_flags(pq, fl, f) for f in ("fold", "h16", "direct")}
    kind_a, kind_s = KINDS[family]
    hk = mod.hk.cpu().double().numpy()
    # analysis
    n0 = pq.launch_count()
    y = mod(x) if flags is None else analysis(mod, x, flags)
    assert pq.launch_count() == n0 + 1
    head = x[:2].clone()
    assert_family(y[:2], {f: analysis(mod, head, v) for f, v in forced.items()}, family)
    assert tiles_per_cta(kind_a, B, F, fl) >= min_tiles, (kind_a, tiles_per_cta(kind_a, B, F, fl))
    if reference:
        assert torch.equal(y, one_tile_per_cta(lambda c: analysis(mod, c, forced[family]), x, kind_a, F, fl))
    check_oracle_analysis(x, y, hk, oracle_excerpts(kind_a, B, F, fl))
    # synthesis
    s = at_offset(y, s_offset)
    n0 = pq.launch_count()
    out = mod.inverse(s) if flags is None else synthesis(mod, s, delay, flags)
    assert pq.launch_count() == n0 + 1
    head = y[:2].clone()
    assert_family(out[:2], {f: synthesis(mod, head, delay, v) for f, v in forced.items()}, family)
    assert tiles_per_cta(kind_s, B, F, fl) >= min_tiles, (kind_s, tiles_per_cta(kind_s, B, F, fl))
    if reference:
        assert torch.equal(out, one_tile_per_cta(lambda c: synthesis(mod, c, delay, forced[family]), y, kind_s, F, fl))
    check_oracle_synthesis(y, out, hk, delay, oracle_excerpts(kind_s, B, F, fl))
    return y, out


# ---------------------------------------------------------------- 1. bank table (no GPU)
def test_bank_table(pq, bank):
    lib = pq._lib
    seen = set()
    for att in ATTENUATIONS:
        mod = bank(att, device="cpu", cls="PQMF")
        L, jlo, kt, fold, h16, residual = N16_TABLE[att]
        assert (mod.hk.shape[1], *taps(mod._flags)) == (L, jlo, kt), att
        assert instantiations(mod) == (fold, h16), att
        no_fold = bool(mod._flags & lib.PQMF_FLAG_NO_FOLD)
        assert no_fold == (mod.fold_residual > FOLD_RESIDUAL_LIMIT), att
        if fold is None:  # Hankel-4 images only: no fold factorisation is attempted
            assert mod.fold_residual == 0.0 and not no_fold and mod.hk.shape[1] != 512
            continue
        assert not no_fold and abs(mod.fold_residual - residual) <= 0.01 * residual, (att, mod.fold_residual)
        seen.add(fold)
        seen.add(h16)
    # what the GPU cases below must keep covering
    assert seen == {(2, 12), (0, 16), (64, 384), (0, 512)}
    assert OTHER_BANKS == [50, 60, 70, 140] and FAMILY_BANKS == [80, 90, 100, 110, 120, 130]
    assert {fold_j(STEADY_T // 16), fold_j(STREAM_PLAN[0] // 16)} == {4, 7}
    assert {fold_j(f) for f in EDGE_FRAMES} == {4, 7} and 160 in EDGE_FRAMES and 161 in EDGE_FRAMES
    assert all(T < 512 and (T // 16) % 2 == 1 for T in EDGE_BLOCKS) and min(STREAM_PLAN) < 512


# ---------------------------------------------------------------- 2. offline steady state, production route
@pytest.mark.gpu
@pytest.mark.parametrize("cls", ["PQMF", "CachedPQMF"])
@pytest.mark.parametrize("att", [100, 120])
def test_offline_steady_state_misaligned(pq, bank, att, cls):
    """1499 rows x 6080 samples: the signal 16 bytes past a 32-byte boundary, the sub-bands 4 bytes past a 16-byte one.  The Hankel-4
    kernels refuse the buffers for their alignment only, so the fold kernels run: ~7.6 analysis and ~10 J = 7 synthesis tiles per CTA."""
    mod = bank(att, cls=cls)
    delay = 1 if cls == "CachedPQMF" else 0
    x0 = signal((STEADY_ROWS, 1, STEADY_T), att)
    x = at_offset(x0, 16)
    assert x.data_ptr() % 32 == 16 and x.contiguous().data_ptr() == x.data_ptr()
    y, out = offline_case(pq, mod, x, delay, "fold", min_tiles=3.0)
    # the aligned call runs the Hankel-4 kernels at this size
    y_al = mod(x0)
    out_al = mod.inverse(y.clone())
    assert not torch.equal(y, y_al)
    assert (y - y_al).abs().max().item() <= 3e-6 and (out - out_al).abs().max().item() <= 8e-6
    # a signal 4 bytes past a 16-byte boundary is refused by the fold kernels too: the direct form
    x4 = at_offset(x0[:3], 4)
    y4 = mod(x4)
    assert torch.equal(y4, analysis(mod, x0[:3], family_flags(pq, mod._flags, "direct")))


# ---------------------------------------------------------------- 3. offline, long rows
@pytest.mark.gpu
@pytest.mark.parametrize("family", ["fold", "h16"])
@pytest.mark.parametrize("cls", ["PQMF", "CachedPQMF"])
@pytest.mark.parametrize("shape", LONG_SHAPES, ids=["64x2^19", "64x(2^19-48)", "2x2^21"])
def test_offline_long_rows(pq, bank, shape, cls, family):
    """Forced fold / Hankel-16 on long rows: 64 x 2^19 (~28 fold analysis tiles per CTA; rows straddle CTAs, so advance() carries),
    the same ragged in tiles, and 2 x 2^21, whose rows are longer than the grid (step_b == 0; no one-tile reference exists)."""
    B, T = shape
    mod = bank(120 if family == "h16" else 100, cls=cls)
    delay = 1 if cls == "CachedPQMF" else 0
    flags = family_flags(pq, mod._flags, family)
    F = T // 16
    x = signal((B, 1, T), B + T)
    ka, ks = KINDS[family]
    wide = B == 2
    if wide:
        for kind in (ka, ks):
            tpr, ctas, _ = launch(kind, F, flags)
            assert tpr > ctas, (kind, tpr, ctas)
    y, out = offline_case(pq, mod, x, delay, family, flags=flags, min_tiles=3.0, reference=not wide)
    # within tolerance of the default (Hankel-4) call on the same input
    assert (y - mod(x)).abs().max().item() <= 3e-6
    assert (out - mod.inverse(y)).abs().max().item() <= 8e-6


# ---------------------------------------------------------------- 4. streaming steady state
def grouped_step(pq, mod, x, xs_in, ss_in, parity_in, parity_out, flags, group=16):
    """stream_step on contiguous groups of <= `group` streams (one tile per CTA): (out, y, new x state, new s state)"""
    outs, ys, xss, sss = [], [], [], []
    hk = mod.hk.float()
    for g in range(0, x.shape[0], group):
        xo, so = torch.empty_like(xs_in[g:g + group]), torch.empty_like(ss_in[g:g + group])
        o, y = torch.ops.pqmf_b200.stream_step(x[g:g + group], hk, mod._tables, xs_in[g:g + group], xo, ss_in[g:g + group], so, parity_in,
                                               parity_out, flags)
        outs.append(o)
        ys.append(y)
        xss.append(xo)
        sss.append(so)
    return torch.cat(outs), torch.cat(ys), torch.cat(xss), torch.cat(sss)


def stream_rows(B, F, flags, family):
    """streams whose tiles are the sampled tiles of both directions (a stream is one tile in each)"""
    rows = set()
    for kind in KINDS[family]:
        tpr, ctas, _ = launch(kind, F, flags)
        rows |= {t // tpr for t in sampled_tiles(B * tpr, min(ctas, B * tpr))}
    return sorted(rows)


def run_stream(pq, mod, family, B, plan, rows, seed, grouped=True, fp32_twin=None, min_tiles=0.0):
    """Blocks of B streams through process_stream (every third block: forward_stream + inverse_stream).  After every block: two launches,
    outputs bit-equal to the grouped one-tile-per-CTA reference with the family's forced flags (on the first block: different bits from
    the other families), both state halves bit-equal to the last 512 samples / 32 frames of history ++ block, `rows` against the float64
    streaming oracle, the fp32 twin (if given) within 3e-6 / 8e-6.  At the end, streamed = offline on the zero-prefixed signal."""
    hk64 = mod.hk.cpu().double().numpy()
    st = O.StreamState(len(rows), 16, 512)
    ridx = torch.tensor(rows, device="cuda")
    xs_prev, ss_prev = torch.zeros(B, 512, device="cuda"), torch.zeros(B, 16, 32, device="cuda")
    forced = {f: family_flags(pq, mod._flags, f) for f in ("fold", "h16", "direct")}
    xs_all, ys_all, outs_all = [], [], []
    for k, T in enumerate(plan):
        F = T // 16
        if k == 0:
            for kind in KINDS[family]:
                assert tiles_per_cta(kind, B, F, mod._flags) >= min_tiles, (kind, tiles_per_cta(kind, B, F, mod._flags))
        x = signal((B, 1, T), seed + k)
        pin, pout = mod._frames_in % 2, mod._frames_out % 2
        n0 = pq.launch_count()
        if k % 3 == 1:
            y = mod.forward_stream(x)
            out = mod.inverse_stream(y)
        else:
            out, y = mod.process_stream(x)
        assert pq.launch_count() == n0 + 2, k
        if grouped:
            for kind in KINDS[family]:
                tpr, ctas, _ = launch(kind, F, mod._flags)
                assert min(16, B) * tpr <= ctas, (kind, F)
            out_r, y_r, _, _ = grouped_step(pq, mod, x, xs_prev, ss_prev.reshape(B, 512), pin, pout, forced[family])
            assert torch.equal(y, y_r) and torch.equal(out, out_r), ("grouped reference", k)
            if k == 0:
                n = min(B, 16)
                calls = {f: grouped_step(pq, mod, x[:n], xs_prev[:n], ss_prev[:n].reshape(n, 512), pin, pout, v) for f, v in forced.items()}
                assert_family(y[:n], {f: c[1] for f, c in calls.items()}, family)
                assert_family(out[:n], {f: c[0] for f, c in calls.items()}, family)
        xs_new = torch.cat([xs_prev, x[:, 0]], -1)[:, -512:].contiguous()
        ss_new = torch.cat([ss_prev, y], -1)[..., -32:].contiguous()
        assert torch.equal(mod._x_state[mod._x_slot], xs_new), ("analysis state", k)
        assert torch.equal(mod._s_state[mod._s_slot].view(B, 16, 32), ss_new), ("synthesis state", k)
        xs_prev, ss_prev = xs_new, ss_new
        y64 = O.stream_analysis(x[ridx, 0].cpu().double().numpy(), hk64, st)
        o64 = O.stream_synthesis(y[ridx].cpu().double().numpy(), hk64, st)
        ea = np.abs(y[ridx].cpu().numpy() - y64).max(axis=(1, 2))
        es = np.abs(out[ridx, 0].cpu().numpy() - o64).max(axis=1)
        assert ea.max() <= TOL / 2, ("analysis", k, rows[int(ea.argmax())], float(ea.max()))
        assert es.max() <= TOL / 2, ("synthesis", k, rows[int(es.argmax())], float(es.max()))
        if fp32_twin is not None:  # each direction on the same input
            y_p = fp32_twin.forward_stream(x)
            out_p = fp32_twin.inverse_stream(y)
            assert (y - y_p).abs().max().item() <= 3e-6 and (out - out_p).abs().max().item() <= 8e-6, k
        xs_all.append(x)
        ys_all.append(y)
        outs_all.append(out)
    x, y_s, out_s = torch.cat(xs_all, -1), torch.cat(ys_all, -1), torch.cat(outs_all, -1)
    t = x.shape[-1]
    assert not mod.streaming  # forward / inverse are the offline calls; they leave the streaming state alone
    y_off = mod(torch.cat([torch.zeros(B, 1, 256, device="cuda"), x], -1))[..., :t // 16]
    assert (y_s - y_off).abs().max().item() <= 2e-6
    out_off = mod.inverse(torch.cat([torch.zeros(B, 16, 16, device="cuda"), y_s], -1))[..., :t]
    assert (out_s - out_off).abs().max().item() <= 4e-6


@pytest.mark.gpu
@pytest.mark.parametrize("family", ["fold", "h16"])
def test_many_streams_48k_blocks(pq, bank, family):
    """4096 streams x 480-sample blocks (and one of 48, one of 960): ~7 fold analysis, ~14 J = 4 fold synthesis tiles per CTA; with
    exact=True the Hankel-16 kernels, ~9 / ~7.  Blocks shorter than L: both rolls read the old history."""
    mod = bank(100, "exact" if family == "h16" else "mod")
    F = STREAM_PLAN[0] // 16
    rows = stream_rows(STREAMS, F, mod._flags, family)
    run_stream(pq, mod, family, STREAMS, STREAM_PLAN, rows, seed=7 + len(family), min_tiles=3.0)


@pytest.mark.gpu
def test_few_streams_long_blocks(pq, bank):
    """2 streams x 2^21-sample blocks on the fold kernels: rows longer than the grid in both directions (step_b == 0).  No one-tile
    reference exists; the fp32 twin, the oracle on both streams and the state bits instead."""
    mod = bank(100)
    T = 1 << 21
    for kind in KINDS["fold"]:
        tpr, ctas, _ = launch(kind, T // 16, mod._flags)
        assert tpr > ctas, (kind, tpr, ctas)
    run_stream(pq, mod, "fold", 2, [T, T], [0, 1], seed=21, grouped=False, fp32_twin=bank(100, "fp32"))
    # the route, on the first block's input from a zero state
    x = signal((2, 1, T), 21)
    z = torch.zeros(2, 512, device="cuda")
    calls = {f: grouped_step(pq, mod, x, z, z, 0, 0, family_flags(pq, mod._flags, f)) for f in ("fold", "h16", "direct")}
    mod.reset_stream()
    out, y = mod.process_stream(x)
    assert_family(y, {f: c[1] for f, c in calls.items()}, "fold")
    assert_family(out, {f: c[0] for f, c in calls.items()}, "fold")


# ---------------------------------------------------------------- 5. StreamGraph
@pytest.mark.gpu
def test_stream_graph_fold_steady_state(pq, bank):
    """StreamGraph replay of 4096 x 480 blocks (the fold kernels at ~7 / ~14 tiles per CTA): bit-equal to eager, across a reset()"""
    streams, block, n_blocks = STREAMS, 480, 5
    x = signal((streams, 1, block * n_blocks), 480)
    eager = bank(100)
    ys, outs = [], []
    for i in range(n_blocks):
        out, y = eager.process_stream(x[..., i * block:(i + 1) * block].contiguous())
        ys.append(y)
        outs.append(out)
    y_e, out_e = torch.cat(ys, -1), torch.cat(outs, -1)
    # the eager blocks ran the fold kernels
    z = torch.zeros(streams, 512, device="cuda")
    _, y_f, _, _ = grouped_step(pq, eager, x[..., :block].contiguous(), z, z, 0, 0, family_flags(pq, eager._flags, "fold"))
    assert torch.equal(y_f, y_e[..., :block // 16])
    assert min(tiles_per_cta(kind, streams, block // 16, eager._flags) for kind in KINDS["fold"]) >= 3.0
    graph = pq.StreamGraph(bank(100, "twin"), streams, block)
    for rep in range(2):
        ys, outs = [], []
        for i in range(n_blocks):
            y, out = graph.step(x[..., i * block:(i + 1) * block])
            ys.append(y.clone())
            outs.append(out.clone())
        assert torch.equal(torch.cat(ys, -1), y_e) and torch.equal(torch.cat(outs, -1), out_e), rep
        graph.reset()


# ---------------------------------------------------------------- 6. every n_band-16 bank
@pytest.mark.gpu
@pytest.mark.parametrize("cls", ["PQMF", "CachedPQMF"])
@pytest.mark.parametrize("att", FAMILY_BANKS)
def test_every_bank_offline(pq, bank, att, cls):
    """467 misaligned rows x 6080 samples, 2-3 tiles per CTA in every family and direction: the fold kernels (default), Hankel-16 via
    exact=True and via the forced flags; PQMF (delay 0) and CachedPQMF (delay 1: off2 = 240, the shift path)."""
    delay = 1 if cls == "CachedPQMF" else 0
    x = at_offset(signal((BANK_ROWS, 1, STEADY_T), att + delay), 16)
    mod = bank(att, cls=cls)
    assert not mod._flags & pq._lib.PQMF_FLAG_NO_FOLD  # factorisable: the fold kernels apply
    offline_case(pq, mod, x, delay, "fold", min_tiles=2.0)
    offline_case(pq, bank(att, "exact", cls=cls), x, delay, "h16", min_tiles=2.0)
    offline_case(pq, mod, x, delay, "h16", flags=family_flags(pq, mod._flags, "h16"), min_tiles=2.0)


@pytest.mark.gpu
@pytest.mark.parametrize("family", ["fold", "h16"])
@pytest.mark.parametrize("att", FAMILY_BANKS)
def test_every_bank_streaming(pq, bank, att, family):
    """1500 lockstep streams x 480-sample blocks (one of 48): 2-3 tiles per CTA at least, in every direction"""
    mod = bank(att, "exact" if family == "h16" else "mod")
    B, plan = 1500, [480, 48, 480]
    rows = stream_rows(B, plan[0] // 16, mod._flags, family)
    run_stream(pq, mod, family, B, plan, rows, seed=att, min_tiles=2.0)


@pytest.mark.gpu
@pytest.mark.parametrize("att", OTHER_BANKS)
def test_other_banks_run_the_direct_form(pq, bank, att):
    """L != 512: no fold or Hankel-16 kernels.  Small offline calls (aligned and misaligned) and streaming blocks are bit-equal to the
    plain-fp32 twin's (the direct form)."""
    for cls in ("PQMF", "CachedPQMF"):
        mod, twin = bank(att, cls=cls), bank(att, "fp32", cls=cls)
        x = signal((3, 1, STEADY_T), att)
        for xv in (x, at_offset(x, 16)):
            y = mod(xv)
            assert torch.equal(y, twin(x))
            assert torch.equal(mod.inverse(at_offset(y, 4)), twin.inverse(y))
    mod, twin = bank(att), bank(att, "fp32")
    for k, T in enumerate([480, 48, 480]):
        x = signal((5, 1, T), att + k)
        out, y = mod.process_stream(x)
        out_t, y_t = twin.process_stream(x)
        assert torch.equal(y, y_t) and torch.equal(out, out_t), k
    assert torch.equal(mod._x_state, twin._x_state) and torch.equal(mod._s_state, twin._s_state)


# ---------------------------------------------------------------- 7. edges
@pytest.mark.gpu
@pytest.mark.parametrize("cls", ["PQMF", "CachedPQMF"])
@pytest.mark.parametrize("n_frames", EDGE_FRAMES)
def test_edge_frame_counts(pq, bank, n_frames, cls):
    """3 rows of F frames, both directions, the fold kernels and (exact=True) Hankel-16: partial tiles, and the J = 4 / J = 7 switch of
    the fold synthesis at F = 160 / 161.  Every frame against the float64 oracle."""
    delay = 1 if cls == "CachedPQMF" else 0
    x = signal((3, 1, 16 * n_frames), n_frames)
    for role, family in (("mod", "fold"), ("exact", "h16")):
        mod = bank(100, role, cls=cls)
        y, out = offline_case(pq, mod, x, delay, family)
        hk = mod.hk.cpu().double().numpy()
        check_oracle_analysis(x, y, hk, [(b, 0, n_frames) for b in range(3)])
        check_oracle_synthesis(y, out, hk, delay, [(b, 0, n_frames) for b in range(3)])


@pytest.mark.gpu
@pytest.mark.parametrize("family", ["fold", "h16"])
@pytest.mark.parametrize("att", [100, 120])
def test_edge_stream_blocks(pq, bank, att, family):
    """blocks of 496, 16 and 48 samples (T < L, odd frame counts: the parity alternates) on 5 streams, every stream against the oracle"""
    mod = bank(att, "exact" if family == "h16" else "mod")
    run_stream(pq, mod, family, 5, EDGE_BLOCKS, list(range(5)), seed=att + 3)


# ---------------------------------------------------------------- 8. 64-bit offsets
@pytest.mark.gpu
def test_64_bit_offsets(pq, bank):
    """2049 misaligned rows x 2^20 samples (> 2^31 elements in x, y and out): the fold kernels; the last rows bit-equal to those rows
    alone, and oracle excerpts on the last row"""
    free, _ = torch.cuda.mem_get_info()
    if free < 40 * 2 ** 30:
        pytest.skip(f"needs 40 GB of free device memory, {free / 2 ** 30:.1f} GB free")
    mod = bank(100, cls="PQMF")
    B, T = 2049, 1 << 20
    F = T // 16
    fold = family_flags(pq, mod._flags, "fold")
    assert B * T > 2 ** 31
    x = torch.empty(B * T + 4 + 64, device="cuda")[4:4 + B * T].view(B, 1, T)
    for i in range(0, B, 256):
        x[i:i + 256] = signal((min(256, B - i), 1, T), i)
    assert x.data_ptr() % 32 == 16
    assert min(tiles_per_cta(kind, B, F, mod._flags) for kind in KINDS["fold"]) >= 3.0
    last = list(range(B - 3, B))
    xl = x[last].clone()
    n0 = pq.launch_count()
    y = mod(x)
    assert pq.launch_count() == n0 + 1
    del x
    yl = y[last].clone()
    s = at_offset(y, 4)
    del y
    out = mod.inverse(s)
    del s
    direct = family_flags(pq, mod._flags, "direct")
    for j, r in enumerate(last):  # each row alone is one tile per CTA in both directions
        assert torch.equal(yl[j:j + 1], analysis(mod, xl[j:j + 1], fold)), r
        assert torch.equal(out[r:r + 1], synthesis(mod, yl[j:j + 1].clone(), 0, fold)), r
    assert not torch.equal(yl[-1:], analysis(mod, xl[-1:], direct))
    assert not torch.equal(out[-1:], synthesis(mod, yl[-1:].clone(), 0, direct))
    hk = mod.hk.cpu().double().numpy()
    ex = [(2, lo, lo + 128) for lo in (0, F // 2, F - 128)]
    check_oracle_analysis(xl, yl, hk, ex)
    check_oracle_synthesis(yl, out[last], hk, 0, ex)
