"""The int16 PCM instantiation of the offline Hankel-4 kernels (H4Io::PCM) where it can go wrong: the steady state of the persistent
loop, the stereo duo walk of the synthesis (a CTA visits the left and then the right row of a tile and stores whole 32-byte groups of
interleaved frames), the 16- and 32-byte loads of mono and stereo frames and the element-wise loads and stores beyond two channels, the
down-mix, the quantiser's saturation and round-half-even ties, every bank the PCM kernels serve, the dispatcher's alignment rules,
the CTA-pair-only instantiations, 64-bit offsets and the host-buffer round trip.  Every case asserts the route the C entry took
(return code and launch count; native means bit-equal to the float32 Hankel call on pcm / 32768, the direct form means bit-equal to
the ``fp32=True`` twin, and the two differ), bit-identity with the float32 twin (synthesis: clamp(round(v * 32768))), and --
independently of the float32 kernels -- agreement of excerpts with the float64 oracle."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import pqmf_oracle as O

pytestmark = pytest.mark.gpu

CLASSES = ["PQMF", "CachedPQMF"]
TOL = 1e-5
TILE = 8192  # samples per tile of the Hankel-4 kernels
ATTENUATIONS = [50, 60, 80, 100, 120, 140]
# banks the host table builder splits into two tap ranges (analysis: two launches; synthesis: the direct form, a split bank's second
# launch accumulates, which int16 cannot), and banks without tables (the direct form both ways)
SPLIT = {(60, 64), (80, 64), (100, 64), (120, 32), (140, 32)}
NO_TABLES = {(120, 64), (140, 64)}


@pytest.fixture(scope="module")
def pq():
    import pqmf_b200

    return pqmf_b200


@pytest.fixture(scope="module")
def bank(pq):
    """modules by (class, attenuation, n_band, exact): the prototype design runs scipy's fmin on the host"""
    cache = {}

    def get(cls, attenuation, n_band, exact=False):
        key = (cls, attenuation, n_band, exact)
        if key not in cache:
            cache[key] = getattr(pq, cls)(attenuation, n_band, exact=exact).cuda()
        return cache[key]

    return get


def audio_pcm(shape, seed):
    """int16 WAV frames [clips, T, C] of audio-like level: N(0, 0.5) clipped to full scale"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    v = (0.5 * torch.randn(shape, generator=g, device="cuda")).clamp_(-1, 1)
    return torch.round(v * 32767.0).to(torch.int16)


def widen(pcm, downmix=False):
    """pcm_sample in torch: v / 32768 per channel [clips, C, T]; the down-mix [clips, 1, T] sums in channel order in fp32, then divides
    by C (a tensor divisor: torch divides by a Python scalar through its reciprocal)"""
    f = pcm.to(torch.float32) / 32768.0
    if not downmix:
        return f.transpose(1, 2).contiguous()
    c = pcm.shape[2]
    if c == 2:
        return ((f[..., 0] + f[..., 1]) / 2)[:, None].contiguous()
    acc = f[..., 0].clone()
    for k in range(1, c):
        acc += f[..., k]
    return (acc / torch.full_like(acc, c))[:, None].contiguous()


def quantise(v, c):
    """float32 rows [clips C, 1, n] -> int16 frames [clips, n, C]: clamp(round half to even(v * 32768))"""
    q = torch.clamp(torch.round(v * 32768.0), -32768, 32767).to(torch.int16)
    return q.view(-1, c, q.shape[-1]).transpose(1, 2).contiguous()


def same_bits(a, b):
    assert a.dtype == b.dtype and a.shape == b.shape, (a.dtype, b.dtype, a.shape, b.shape)
    if a.dtype == torch.float32:
        return torch.equal(a.view(torch.int32), b.view(torch.int32))
    return torch.equal(a, b)


def tables_ptr(mod):
    return mod._tables.data_ptr() if mod._tables.numel() else None


def stream():
    return torch.cuda.current_stream().cuda_stream


def taps(flags):
    """(jlo, kt) of the bank's Hankel-4 images (PQMF_FLAG_TAPS)"""
    return 32 * ((flags >> 8) & 0xF), 32 * ((flags >> 12) & 0x1F)


def f32_analysis(mod, x, flags):
    return torch.ops.pqmf_b200.analysis(x, mod.hk, mod._tables, x.shape[-1] // mod.n_band, flags)


def f32_synthesis(mod, s, delay, flags):
    return torch.ops.pqmf_b200.synthesis(s, mod.hk, mod._tables, delay, flags)


# ---------------------------------------------------------------- the C entries, their route and their float32 twins
def check_analysis(pq, mod, pcm, downmix, native, launches=1, flags=None, y=None):
    """pqmf_analysis_pcm16 on pcm [clips, T, C] (any view) into y [rows, M, F] (fresh, or a view): returns 0 after `launches` launches
    and is bit-equal to the float32 call on the widened rows -- the Hankel call where `native`, the fp32=True twin otherwise."""
    from pqmf_b200 import _lib

    flags = mod._flags if flags is None else flags
    clips, t, c = pcm.shape
    m, length = mod.hk.shape
    rows = clips if downmix else clips * c
    if y is None:
        y = torch.empty(rows, m, t // m, device="cuda")
    n0 = pq.launch_count()
    rc = _lib.cabi.pqmf_analysis_pcm16(pcm.data_ptr(), y.data_ptr(), mod.hk.data_ptr(), tables_ptr(mod), clips, t, c, int(downmix), t // m, m,
                                       length, flags, stream())
    torch.cuda.synchronize()
    assert (rc, pq.launch_count() - n0) == (0, launches)
    x = widen(pcm, downmix)
    hankel = f32_analysis(mod, x, flags).view(y.shape)
    direct = f32_analysis(mod, x, flags | _lib.PQMF_FLAG_FP32).view(y.shape)
    if mod._tables.numel():
        assert not same_bits(hankel, direct)  # the route check has teeth
    assert same_bits(y, hankel if native else direct)
    return y, x.view(rows, t)


def check_synthesis(pq, mod, s, c, delay, native, flags=None, out=None):
    """pqmf_synthesis_pcm16 on s [clips C, M, F] into out [clips, M F, C] (fresh, or a view): returns 0 after one launch and is
    bit-equal to clamp(round(v * 32768)) of the float32 call on the same sub-bands -- the Hankel call where `native`, else the fp32=True
    twin.  Returns out and the float32 values the kernel quantised."""
    from pqmf_b200 import _lib

    flags = mod._flags if flags is None else flags
    rows, m, f = s.shape
    clips = rows // c
    length = mod.hk.shape[1]
    if out is None:
        out = torch.empty(clips, m * f, c, dtype=torch.int16, device="cuda")
    n0 = pq.launch_count()
    rc = _lib.cabi.pqmf_synthesis_pcm16(s.data_ptr(), out.data_ptr(), mod.hk.data_ptr(), tables_ptr(mod), clips, c, f, m, length, delay, flags,
                                        stream())
    torch.cuda.synchronize()
    assert (rc, pq.launch_count() - n0) == (0, 1)
    sc = s.clone()  # the twins read an aligned copy
    hankel = f32_synthesis(mod, sc, delay, flags)
    direct = f32_synthesis(mod, sc, delay, flags | _lib.PQMF_FLAG_FP32)
    if mod._tables.numel():
        assert not same_bits(hankel, direct)
    v = hankel if native else direct
    assert same_bits(out, quantise(v, c))
    return out, v


# ---------------------------------------------------------------- the float64 oracle on excerpts
def oracle_excerpt(x_row, y_row, q_row, hk, delay, start, n, gain=1.0):
    """Frames [start, start + n) of one row's sub-bands and the output samples of those frames, against the float64 oracle run on the
    cropped input they depend on: one filter length of halo on each side, cut at an even frame (the sign mask follows the global frame
    parity), or at the row's own ends.  Analysis: within TOL / 2 of the oracle on the widened row.  Synthesis, on the sub-bands the
    kernel read: |q - clamp(o64 * 32768)| <= 0.5 + 32768 tol (the float bound, then the rounding to an integer); the float bound holds
    for signals up to full scale and grows with `gain` for sub-bands scaled beyond it."""
    m, length = hk.shape
    n_frames = y_row.shape[1]
    halo = length // m
    f0 = max(0, start - halo) & ~1
    f1 = min(n_frames, start + n + halo)
    tol_s = gain * (TOL if m == 64 else TOL / 2)  # n_band 64 synthesis: fp32 accumulation alone is ~4e-6
    if x_row is not None:
        y64 = O.analysis(x_row[f0 * m:f1 * m][None], hk)[0]
        err = np.abs(y_row[:, start:start + n] - y64[:, start - f0:start - f0 + n]).max()
        assert err <= TOL / 2, f"analysis, frames {start}+{n}: |error| {err:.3g}"
    if q_row is not None:
        o64 = O.synthesis(y_row[:, f0:f1][None], hk, delay_frames=delay)[0]
        a = (start - f0) * m
        ref = np.clip(o64[a:a + n * m] * 32768.0, -32768.0, 32767.0)
        err = np.abs(q_row[start * m:(start + n) * m] - ref).max()
        assert err <= 0.5 + 32768 * tol_s, f"synthesis, frames {start}+{n}: |error| {err:.3g} LSB"


def oracle_rows(mod, x, y, q, delay, rows, gain=1.0):
    """Excerpts of the given rows (row = clip C + channel): the row start, tile boundaries (the second tile, one in the middle, the
    last) and the row end.  x [rows, T] widened signal or None, y [rows, M, F], q [clips, M F, C] int16 or None."""
    hk = mod.hk.cpu().double().numpy()
    m = hk.shape[0]
    n_frames = y.shape[-1]
    c = q.shape[2] if q is not None else 1
    n = 4096 // m  # frames of 4096 samples: half a tile
    fpt = TILE // m
    tiles_per_row = -(-n_frames * m // TILE)
    starts = [0, fpt - n // 2, (tiles_per_row // 2) * fpt - n // 2, (tiles_per_row - 1) * fpt - n // 2, n_frames - n]
    for r in rows:
        xr = x[r].double().cpu().numpy() if x is not None else None
        yr = y[r].double().cpu().numpy()
        qr = q[r // c, :, r % c].double().cpu().numpy() if q is not None else None
        for s in starts:
            oracle_excerpt(xr, yr, qr, hk, delay, s, n, gain)


def delay_of(cls):
    return 1 if cls == "CachedPQMF" else 0


# ---------------------------------------------------------------- 1. steady state of the persistent loop
# 37 clips x (33 tiles - 12 frames): 1221 tiles a row set, odd, ~8 per CTA on 148 SMs, with a partial last tile; T % 8 == 0 and
# F % 4 == 0, so both directions run natively.  Stereo: 2442 analysis tiles, and the duo walk's 1221 (clip, tile) pairs of two visits.
def steady_shape(m, c):
    return (37, 33 * TILE - 12 * m, c)


@pytest.mark.parametrize("cls", CLASSES)
@pytest.mark.parametrize("n_band", [4, 8, 16, 32])
def test_steady_state_mono(pq, bank, n_band, cls):
    mod = bank(cls, 100, n_band)
    pcm = audio_pcm(steady_shape(n_band, 1), seed=n_band)
    y, x = check_analysis(pq, mod, pcm, False, native=True)
    q, _ = check_synthesis(pq, mod, y, 1, delay_of(cls), native=True)
    oracle_rows(mod, x, y, q, delay_of(cls), rows=(0, 18, 36))


@pytest.mark.parametrize("cls", CLASSES)
@pytest.mark.parametrize("n_band", [4, 8, 16, 32])
def test_steady_state_stereo(pq, bank, n_band, cls):
    mod = bank(cls, 100, n_band)
    pcm = audio_pcm(steady_shape(n_band, 2), seed=100 + n_band)
    y, x = check_analysis(pq, mod, pcm, False, native=True)
    q, _ = check_synthesis(pq, mod, y, 2, delay_of(cls), native=True)
    oracle_rows(mod, x, y, q, delay_of(cls), rows=(0, 1, 36, 37, 72, 73))  # both channels of the first, a middle and the last clip
    yd, xd = check_analysis(pq, mod, pcm, True, native=True)
    oracle_rows(mod, xd, yd, None, 0, rows=(0, 18, 36))


# ---------------------------------------------------------------- 2. every bank the PCM kernels serve
# 7 stereo clips x (29 tiles - 8 frames): 406 analysis tiles (2-3 per CTA), 203 for the down-mix, and 203 (clip, tile) pairs of two
# visits for the synthesis.  n_band 4 runs both classes: their synthesis offsets select the two synthesis images
# (test_n_band_4_sweep_hits_both_synthesis_images); other band counts alternate the class over the sweep.
def sweep():
    cases = []
    for i, att in enumerate(ATTENUATIONS):
        for j, m in enumerate([4, 8, 16, 32, 64]):
            cases += [(att, m, cls, False) for cls in (CLASSES if m == 4 else [CLASSES[(i + j) % 2]])]
    return cases + [(60, 4, "CachedPQMF", True), (100, 16, "PQMF", True), (80, 32, "CachedPQMF", True)]


@pytest.mark.parametrize("attenuation,n_band,cls,exact", sweep())
def test_every_bank(pq, bank, attenuation, n_band, cls, exact):
    mod = bank(cls, attenuation, n_band, exact)
    tables = (attenuation, n_band) not in NO_TABLES
    split = (attenuation, n_band) in SPLIT
    assert (mod._tables.numel() > 0) == tables and bool(mod._flags & pq._lib.PQMF_FLAG_H4_SPLIT) == split
    assert bool(mod._flags & pq._lib.PQMF_FLAG_EXACT) == exact
    pcm = audio_pcm((7, 29 * TILE - 8 * n_band, 2), seed=attenuation + n_band)
    y, x = check_analysis(pq, mod, pcm, False, native=tables, launches=2 if split else 1)
    q, _ = check_synthesis(pq, mod, y, 2, delay_of(cls), native=tables and not split)
    oracle_rows(mod, x, y, q, delay_of(cls), rows=(0, 7, 13))
    yd, xd = check_analysis(pq, mod, pcm, True, native=tables, launches=2 if split else 1)
    oracle_rows(mod, xd, yd, None, 0, rows=(6,))


def test_bank_table(pq, bank):
    """The split / no-table status the sweep above relies on, so that it cannot go vacuous when the trim or split logic changes."""
    for att in ATTENUATIONS:
        for m in [4, 8, 16, 32, 64]:
            mod = bank("PQMF", att, m)
            length = mod.hk.shape[1]
            routed = pq._lib.cabi.pqmf_path_for(m, length, tables_ptr(mod), mod._flags)
            if (att, m) in NO_TABLES:
                assert mod._tables.numel() == 0 and routed == 0, (att, m)
            else:
                assert routed == 1 and bool(mod._flags & pq._lib.PQMF_FLAG_H4_SPLIT) == ((att, m) in SPLIT), (att, m)


def test_n_band_4_sweep_hits_both_synthesis_images(bank):
    """n_band 4 has two synthesis images; the router picks variant (o - ehi) & 1 (o = synthesis offset in frames, ehi = largest
    frame lag with a tap).  The sweep must run both."""
    seen = set()
    for att in ATTENUATIONS:
        for delay, cls in enumerate(CLASSES):
            mod = bank(cls, att, 4)
            jlo, kt = taps(mod._flags)
            o = mod.hk.shape[1] // 8 - delay
            seen.add((o - ((jlo + kt) // 4 - 1)) & 1)
    assert seen == {0, 1}


# ---------------------------------------------------------------- 3. more than two channels on the Hankel kernels
# 11 clips x (9 tiles - 4 frames): C x 99 analysis tiles, 99 for the down-mix: the element-wise loads (pcm_sample, either the channel
# or the down-mix) and, in synthesis, pcm_store8's element-wise stores.
@pytest.mark.parametrize("n_band,channels", [(16, 3), (8, 5), (32, 6), (4, 3)])
def test_many_channels(pq, bank, n_band, channels):
    mod = bank("CachedPQMF", 100, n_band)
    pcm = audio_pcm((11, 9 * TILE - 4 * n_band, channels), seed=channels * n_band)
    y, x = check_analysis(pq, mod, pcm, False, native=True)
    q, _ = check_synthesis(pq, mod, y, channels, 1, native=True)
    oracle_rows(mod, x, y, q, 1, rows=(0, channels - 1, 11 * channels - 1))
    yd, xd = check_analysis(pq, mod, pcm, True, native=True)
    oracle_rows(mod, xd, yd, None, 0, rows=(0, 10))


# ---------------------------------------------------------------- 4. the quantiser's edges
# Sub-bands of a loud signal, scaled so that the synthesis clips at both ends.  The compared data must contain saturated samples at
# +32767 and -32768 and exact ties (v * 32768 with a fractional part of exactly 0.5, about 2^-9 of the samples near full scale) where
# round-half-even and round-half-away differ.
@pytest.mark.parametrize("n_band,channels,native", [(16, 1, True), (8, 2, True), (32, 3, True), (64, 1, False)])
def test_quantiser_edges(pq, bank, n_band, channels, native):
    mod = bank("PQMF", 100, n_band)  # n_band 64 at attenuation 100 is split: the direct form's quantiser
    pcm = audio_pcm((13, 9 * TILE, channels), seed=7 * n_band)
    y = mod.forward_pcm16(pcm).view(13 * channels, n_band, -1) * 1.9
    q, v = check_synthesis(pq, mod, y, channels, 0, native=native)
    assert bool((q == 32767).any()) and bool((q == -32768).any())
    w = v * 32768.0  # exact
    tie = ((w - torch.floor(w)) == 0.5) & (w.abs() < 32767)
    away = torch.trunc(w + 0.5 * torch.sign(w))
    assert int(tie.sum()) > 100 and bool((tie & (torch.round(w) != away)).any())
    oracle_rows(mod, None, y, q, 0, rows=(0, 13 * channels - 1), gain=1.9)


# ---------------------------------------------------------------- 5. alignment and guards (C ABI)
GUARD = 64  # bytes of sentinel on each side of every view


def guarded(numel, dtype, offset_bytes):
    """a view of `numel` elements `offset_bytes` past a 32-byte boundary inside a buffer whose margins hold a sentinel"""
    size = torch.empty(0, dtype=dtype).element_size()
    start = (GUARD + offset_bytes) // size
    buf = torch.full((numel + 2 * GUARD // size + offset_bytes // size,), -12345 if dtype == torch.int16 else 1234.5, dtype=dtype, device="cuda")
    view = buf[start:start + numel]
    assert view.data_ptr() % 32 == offset_bytes % 32
    return buf, view, start


def guards_hold(buf, start, numel):
    sentinel = -12345 if buf.dtype == torch.int16 else 1234.5
    return bool((buf[:start] == sentinel).all()) and bool((buf[start + numel:] == sentinel).all())


# (direction, channels, offset of the PCM buffer, offset of the sub-band buffer, native).  13 clips of 8 tiles: 104 (mono) or 208
# (stereo) tiles.  PCM input needs 32 bytes, sub-bands 16, mono and element-wise PCM output 16, interleaved stereo output 32 (the duo
# drain's 32-byte stores).
ALIGNMENT = [
    ("analysis", 2, 2, 0, False),
    ("analysis", 1, 16, 0, False),
    ("analysis", 2, 16, 0, False),
    ("analysis", 1, 32, 0, True),
    ("analysis", 2, 32, 0, True),
    ("analysis", 2, 0, 4, False),
    ("synthesis", 2, 0, 4, False),
    ("synthesis", 1, 16, 0, True),
    ("synthesis", 2, 16, 0, False),
    ("synthesis", 2, 32, 0, True),
    ("synthesis", 1, 2, 0, False),
    ("synthesis", 2, 2, 0, False),
    ("synthesis", 3, 16, 0, True),
]


@pytest.mark.parametrize("direction,channels,pcm_offset,bands_offset,native", ALIGNMENT)
def test_alignment(pq, bank, direction, channels, pcm_offset, bands_offset, native):
    mod = bank("PQMF", 100, 16)
    clips, t = 13, 8 * TILE
    src = audio_pcm((clips, t, channels), seed=channels + pcm_offset)
    n_pcm, n_bands = src.numel(), clips * channels * t
    bands_shape = (clips * channels, 16, t // 16)
    if direction == "analysis":
        pbuf, pview, ps = guarded(n_pcm, torch.int16, pcm_offset)
        pview.copy_(src.view(-1))
        ybuf, yview, ys = guarded(n_bands, torch.float32, bands_offset)
        y, _ = check_analysis(pq, mod, pview.view(src.shape), False, native, y=yview.view(bands_shape))
        assert guards_hold(ybuf, ys, n_bands) and guards_hold(pbuf, ps, n_pcm)
        assert same_bits(y, mod.forward_pcm16(src).view(bands_shape)) == native  # the torch op's fresh buffers: native
    else:
        y = mod.forward_pcm16(src).view(bands_shape)
        sbuf, sview, ss = guarded(n_bands, torch.float32, bands_offset)
        sview.copy_(y.reshape(-1))
        obuf, oview, os_ = guarded(n_pcm, torch.int16, pcm_offset)
        check_synthesis(pq, mod, sview.view(bands_shape), channels, 0, native, out=oview.view(src.shape))
        assert guards_hold(obuf, os_, n_pcm) and guards_hold(sbuf, ss, n_bands)


# ---------------------------------------------------------------- 6. PQMF_FLAG_NO_PAIR
def test_no_pair(pq, bank):
    """The PCM instantiations exist as CTA pairs only: with PQMF_FLAG_NO_PAIR the PCM calls come back through the direct form (rc 0,
    one launch), while the float32 calls run the single-CTA Hankel kernels (not the direct form's bits)."""
    from pqmf_b200 import _lib

    mod = bank("CachedPQMF", 100, 16)
    flags = mod._flags | _lib.PQMF_FLAG_NO_PAIR
    for c in (1, 2):
        pcm = audio_pcm((13, 8 * TILE, c), seed=50 + c)
        y, _ = check_analysis(pq, mod, pcm, False, native=False, flags=flags)
        check_synthesis(pq, mod, y, c, 1, native=False, flags=flags)
        assert not same_bits(y, mod.forward_pcm16(pcm).view(y.shape))  # the paired PCM kernels run without the flag


# ---------------------------------------------------------------- 7. 64-bit offsets
@pytest.mark.parametrize("channels,clips", [(1, 4097), (2, 2049)])
def test_64_bit_offsets(pq, bank, channels, clips):
    """Clips of 2^19 samples at n_band 16: more than 2^31 int16 elements in and out and more than 2^32 bytes of sub-bands; the last
    clip starts beyond either limit (stereo: the duo stores of the last clips).  About 17 GB of device memory."""
    free, _ = torch.cuda.mem_get_info()
    if free < 24 * 2 ** 30:
        pytest.skip(f"needs 24 GB of free device memory, {free / 2 ** 30:.1f} GB free")
    mod = bank("PQMF", 100, 16)
    t = 1 << 19
    pcm = torch.empty(clips, t, channels, dtype=torch.int16, device="cuda")
    for r0 in range(0, clips, 512):
        pcm[r0:r0 + 512] = audio_pcm((min(512, clips - r0), t, channels), seed=r0)
    assert pcm.numel() > 2 ** 31 and pcm.numel() * 4 > 2 ** 32
    ends = [0, 1, clips - 2, clips - 1]
    pcm_ends = pcm[ends].contiguous()
    y = mod.forward_pcm16(pcm)
    del pcm
    q = mod.inverse_pcm16(y)
    # two clips are 128 (mono) or 256 (stereo) tiles: the same kernels run them as a separate call
    for k in (slice(0, 2), slice(2, 4)):
        y_sep, x_sep = check_analysis(pq, mod, pcm_ends[k], False, native=True)
        assert same_bits(y_sep, y[ends[k]].view(y_sep.shape))
        q_sep, _ = check_synthesis(pq, mod, y_sep, channels, 0, native=True)
        assert same_bits(q_sep, q[ends[k]])
    oracle_rows(mod, x_sep, y_sep, q_sep, 0, rows=(2 * channels - 1,))
    del y, q
    torch.cuda.empty_cache()


# ---------------------------------------------------------------- 8. the host-buffer round trip
# (class, attenuation, n_band, clips, T, C, chunk plan at the default chunk size): ramp chunks at both ends and a last chunk that
# absorbed an undersized remainder
HOST = [
    ("CachedPQMF", 100, 16, 61, 65536, 2, [6, 8, 8, 16, 16, 7]),
    ("CachedPQMF", 100, 64, 101, 65536, 1, [12, 16, 16, 32, 25]),  # split bank: two analysis launches, the synthesis' direct form
    ("PQMF", 100, 4, 145, 32768, 1, [24, 32, 32, 32, 25]),
    ("CachedPQMF", 100, 8, 40, 40960, 3, [7, 8, 8, 8, 9]),
]


@pytest.mark.parametrize("cls,attenuation,n_band,clips,t,channels,plan", HOST)
def test_roundtrip_host(pq, bank, cls, attenuation, n_band, clips, t, channels, plan):
    """pqmf_roundtrip_host_pcm16 runs pqmf_analysis_pcm16 / pqmf_synthesis_pcm16 per chunk of whole clips: bit-equal to one device call
    per direction, since every chunk keeps the route (at least 96 tiles) and a tile's result does not depend on the CTA that runs it."""
    from pqmf_b200 import _lib

    f = _lib.cabi.pqmf_host_chunk_plan
    f.restype = ctypes.c_int
    f.argtypes = [ctypes.c_int, ctypes.c_long, ctypes.c_int, ctypes.POINTER(ctypes.c_long), ctypes.c_int]
    n = f(clips, t, channels, None, 0)
    buf = (ctypes.c_long * n)()
    f(clips, t, channels, buf, n)
    assert list(buf) == plan
    mod = bank(cls, attenuation, n_band)
    split = (attenuation, n_band) in SPLIT
    delay = delay_of(cls)
    pcm = audio_pcm((clips, t, channels), seed=clips)
    y, _ = check_analysis(pq, mod, pcm, False, native=True, launches=2 if split else 1)
    q, _ = check_synthesis(pq, mod, y, channels, delay, native=not split)
    hp = pcm.cpu().pin_memory()
    ho = torch.empty_like(hp).pin_memory()
    hy = torch.empty(clips * channels, n_band, t // n_band).pin_memory()
    hk_h, tab_h = mod.hk.cpu().contiguous(), mod._tables.cpu().contiguous()
    rc = _lib.cabi.pqmf_roundtrip_host_pcm16(hp.data_ptr(), hy.data_ptr(), ho.data_ptr(), hk_h.data_ptr(), tab_h.data_ptr(), clips, t, channels,
                                             n_band, hk_h.shape[1], delay, int(mod._flags), torch.cuda.current_device())
    assert rc == 0, _lib.strerror(rc)
    assert same_bits(hy, y.cpu()) and same_bits(ho, q.cpu())
    _lib.cabi.pqmf_host_release()
