"""GPU parity: the CUDA path (through the C ABI and through the torch ops / module API) against the
oracle and the reference-generated golden vectors.  Tolerance: north_star's max-abs <= 1e-5 against the
reference's fp32 results, round-trip SNR within 0.1 dB."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import pqmf_oracle as O

pytestmark = pytest.mark.gpu

TOL = 1e-5  # BASELINE.json north_star: max-abs error vs the reference's own fp32 PQMF


@pytest.fixture(scope="module")
def pq():
    import pqmf_b200

    return pqmf_b200


@pytest.fixture(scope="module")
def lib():
    from pqmf_b200 import _lib

    return _lib


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _tables_for(lib, hk, h):
    tables, res, fast_flags = lib.build_tables(torch.from_numpy(hk), torch.from_numpy(h))
    return (tables.cuda(), fast_flags) if tables.numel() else (None, 0)


# ------------------------------------------------------------------ raw C ABI (ctypes, device pointers)
@pytest.mark.parametrize("m", (4, 8, 16, 32, 64))
@pytest.mark.parametrize("exact", (True, False))
def test_cabi_offline_vs_golden(golden, lib, m, exact):
    g = golden(f"vectors_M{m}.npz")
    bank = golden(f"bank_M{m}.npz")
    hk, h = bank["hk"], bank["h"]
    length = hk.shape[1]
    x = g["x"][:, 0]
    b, t = x.shape
    d_x, d_hk = dev(x), dev(hk)
    tables, fast_flags = (None, 0) if exact else _tables_for(lib, hk, h)
    flags = lib.PQMF_FLAG_EXACT if exact else fast_flags
    tp = tables.data_ptr() if tables is not None else None
    y = torch.empty(b, m, t // m, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    rc = lib.cabi.pqmf_analysis_f32(d_x.data_ptr(), y.data_ptr(), d_hk.data_ptr(), tp, b, t, t // m, m, length, flags, st)
    assert rc == 0, lib.strerror(rc)
    torch.cuda.synchronize()
    for key in ("y_poly", "y_classic", "y_cached"):
        assert np.abs(y.cpu().numpy() - g[key]).max() <= TOL, key
    # synthesis is fed the REFERENCE's sub-bands (SURVEY 8d parity protocol)
    s = dev(g["y_poly"])
    for delay, key in ((0, "out_poly"), (1, "out_cached")):
        out = torch.empty(b, t, device="cuda")
        rc = lib.cabi.pqmf_synthesis_f32(s.data_ptr(), out.data_ptr(), d_hk.data_ptr(), tp, b, t // m, m, length, delay, flags, st)
        assert rc == 0, lib.strerror(rc)
        torch.cuda.synchronize()
        assert np.abs(out.cpu().numpy() - g[key][:, 0]).max() <= TOL, key


def test_cabi_rejects_bad_arguments(lib):
    c = lib.cabi
    assert c.pqmf_analysis_f32(None, None, None, None, 1, 64, 4, 16, 512, 0, None) == -1
    assert c.pqmf_analysis_f32(None, None, None, None, 1, 64, 4, 1, 512, 0, None) == -1
    assert c.pqmf_synthesis_f32(None, None, None, None, 1, 4, 16, 512, 2, 0, None) == -1
    assert c.pqmf_analysis_stream_f32(None, None, None, None, None, None, 1, 65, 16, 512, 0, 0, None) == -1
    assert c.pqmf_analysis_f32(None, None, None, None, 0, 64, 4, 16, 512, 0, None) == 0  # empty batch is a no-op


# ------------------------------------------------------------------ module API, offline
@pytest.mark.parametrize("m", (4, 8, 16, 32, 64))
@pytest.mark.parametrize("polyphase", (True, False))
def test_module_matches_reference(golden, pq, m, polyphase):
    g = golden(f"vectors_M{m}.npz")
    mod = pq.PQMF(100, m, polyphase=polyphase).cuda()
    assert np.abs(mod.hk.cpu().numpy() - golden(f"bank_M{m}.npz")["hk"]).max() <= 1e-8
    x = dev(g["x"])
    y = mod(x)
    assert y.shape == (2, m, x.shape[-1] // m)
    assert np.abs(y.cpu().numpy() - g["y_poly" if polyphase else "y_classic"]).max() <= TOL
    out = mod.inverse(dev(g["y_poly"]))
    assert out.shape == x.shape
    assert np.abs(out.cpu().numpy() - g["out_poly" if polyphase else "out_classic"]).max() <= TOL
    # round trip through our own sub-bands: SNR within 0.1 dB of the reference's round trip
    rt = mod.inverse(y).cpu().numpy()
    ref_rt = g["out_poly"]
    assert abs(O.snr_db(g["x"], rt) - O.snr_db(g["x"], ref_rt)) <= 0.1


@pytest.mark.parametrize("m", (4, 16, 64))
def test_exact_mode_on_unit_variance_subbands(golden, pq, m):
    g = golden(f"vectors_M{m}.npz")
    mod = pq.PQMF(100, m, exact=True).cuda()
    out = mod.inverse(dev(g["s_rand"]))
    # unit-variance sub-bands give outputs of magnitude ~n_band: the budget scales with the output range
    # (the reference's own fp32 run is ~2e-6 * n_band away from float64 here)
    assert np.abs(out.cpu().numpy() - g["out_rand"]).max() <= TOL * max(1.0, float(np.abs(g["out_rand"]).max()))


@pytest.mark.parametrize("m", (4, 8, 16, 32, 64))
def test_cached_module_and_ragged_lengths(golden, pq, m):
    g = golden(f"vectors_M{m}.npz")
    mod = pq.CachedPQMF(100, m).cuda()
    x = dev(g["x"])
    assert np.abs(mod(x).cpu().numpy() - g["y_cached"]).max() <= TOL
    assert np.abs(mod.inverse(dev(g["y_poly"])).cpu().numpy() - g["out_cached"]).max() <= TOL
    tr = int(g["x_ragged_len"])
    xr = x[..., :tr].contiguous()
    yr = mod(xr)
    assert yr.shape[-1] == -(-tr // m)
    assert np.abs(yr.cpu().numpy() - g["yr_cached"]).max() <= TOL
    classic = pq.PQMF(100, m, polyphase=False).cuda()
    yc = classic(xr)
    assert yc.shape[-1] == tr // m
    assert np.abs(yc.cpu().numpy() - g["yr_classic"]).max() <= TOL
    with pytest.raises(RuntimeError):
        pq.PQMF(100, m).cuda()(xr)  # polyphase needs T % M == 0 (reference: einops error)


def test_torchscript_archive_vectors(golden, pq):
    g = golden("ts_M16.npz")
    mod = pq.CachedPQMF(100, 16).cuda()
    assert np.array_equal(mod.h.cpu().numpy(), g["h"])
    assert tuple(mod.forward_conv.weight.shape) == tuple(g["fwd_weight_shape"])
    assert np.abs(mod.inverse_conv.weight.cpu().numpy() - g["inv_weight"]).max() <= 1e-8
    assert np.abs(mod(dev(g["x"])).cpu().numpy() - g["y"]).max() <= TOL
    assert np.abs(mod.inverse(dev(g["y"])).cpu().numpy() - g["out"]).max() <= TOL


def test_non_power_of_two_classic(golden, pq):
    g = golden("vectors_M12_classic.npz")
    with pytest.raises(AssertionError):
        pq.PQMF(100, 12)
    mod = pq.PQMF(100, 12, polyphase=False).cuda()
    y = mod(dev(g["x"]))
    assert np.abs(y.cpu().numpy() - g["y"]).max() <= TOL
    # the reference's classic synthesis for L % M != 0 follows the same closed form
    out = mod.inverse(dev(g["y"]))
    assert np.abs(out.cpu().numpy() - g["out"]).max() <= TOL


def test_free_functions_skip_the_sign_mask(golden, pq):
    g = golden("vectors_M16.npz")
    hk = dev(golden("bank_M16.npz")["hk"])
    x = dev(g["x"])
    y = pq.reverse_half(pq.polyphase_forward(x, hk))
    assert np.abs(y.cpu().numpy() - g["y_poly"]).max() <= TOL
    y2 = pq.reverse_half(pq.classic_forward(x, hk))
    assert np.abs(y2.cpu().numpy() - g["y_classic"]).max() <= TOL
    s = pq.reverse_half(dev(g["y_poly"]))
    assert np.abs(pq.polyphase_inverse(s, hk).cpu().numpy() - g["out_poly"]).max() <= TOL
    assert np.abs(pq.classic_inverse(s, hk).cpu().numpy() - g["out_classic"]).max() <= TOL
    # pre-arranged filters (rearrange_filter=False) as the reference's callers may pass them
    w = hk.reshape(16, 32, 16).permute(0, 2, 1).contiguous()
    assert torch.equal(pq.polyphase_forward(x, w, rearrange_filter=False), pq.polyphase_forward(x, hk))
    wi = hk.flip(-1).reshape(16, 32, 16).permute(2, 0, 1).contiguous()
    assert torch.equal(pq.polyphase_inverse(s, wi, rearrange_filter=False), pq.polyphase_inverse(s, hk))


def test_flute_config1(golden, pq):
    """BASELINE config 1: audio/flute.wav, n_band 16, attenuation 100, batch 1, padded as the wrappers do."""
    g = golden("flute_C1.npz")
    n_pad = int(g["n_pad"])
    x = np.zeros((1, 1, n_pad), np.float32)
    x[0, 0, : g["pcm"].shape[0]] = g["pcm"].astype(np.float32) / 32768.0
    mod = pq.PQMF(100, 16).cuda()
    y = mod(dev(x))
    out = mod.inverse(y)
    yn, on = y.cpu().numpy(), out.cpu().numpy()
    lo, hi = g["excerpt"]
    assert np.abs(yn[:, :, lo // 16 : hi // 16] - g["y_excerpt"]).max() <= TOL
    assert np.abs(yn[:, :, :64] - g["y_head"]).max() <= TOL
    assert np.abs(on[:, :, lo:hi] - g["out_excerpt"]).max() <= TOL
    assert np.abs(on[:, :, :1024] - g["out_head"]).max() <= TOL
    assert np.abs(on[:, :, -1024:] - g["out_tail"]).max() <= TOL
    assert abs(O.snr_db(x, on) - float(g["flute_M16"])) <= 0.1
    # whole clip against the oracle
    hk = golden("bank_M16.npz")["hk"]
    y64 = O.analysis(x[:, 0], hk)
    assert np.abs(yn - y64).max() <= TOL
    assert np.abs(on[:, 0] - O.synthesis(yn, hk)).max() <= TOL
    cached = pq.CachedPQMF(100, 16).cuda()
    oc = cached.inverse(cached(dev(x))).cpu().numpy()
    assert abs(O.snr_db(x[..., :-16], oc[..., 16:]) - float(g["flute_M16_cached_delay16"])) <= 0.1


# ------------------------------------------------------------------ larger seeded inputs vs the oracle
@pytest.mark.parametrize("m,b,t", ((16, 3, 65536), (16, 1, 16 * 4097), (16, 2, 2048), (16, 5, 48), (8, 2, 40000), (32, 2, 32768)))
def test_against_oracle_various_shapes(golden, pq, m, b, t):
    hk = golden(f"bank_M{m}.npz")["hk"]
    x = O.audio_like((b, 1, t), 4242 + t)
    mod = pq.PQMF(100, m).cuda()
    y = mod(dev(x)).cpu().numpy()
    y64 = O.analysis(x[:, 0], hk)
    assert np.abs(y - y64).max() <= TOL / 2
    s = y64.astype(np.float32)
    out = mod.inverse(dev(s)).cpu().numpy()
    assert np.abs(out[:, 0] - O.synthesis(s, hk)).max() <= TOL / 2


def test_multichannel_is_folded_into_batch(golden, pq):
    g = golden("flutemulti_excerpt.npz")
    x = (g["pcm"].astype(np.float32) / 32768.0)[None]  # [1, 2, T]
    mod = pq.PQMF(100, 16).cuda()
    y = mod(dev(x))
    assert y.shape == (1, 32, x.shape[-1] // 16)
    y_rows = mod(dev(x.reshape(2, 1, -1)))
    assert torch.equal(y.reshape(2, 16, -1), y_rows)
    out = mod.inverse(y)
    assert out.shape == x.shape


def test_empty_and_tiny_inputs(pq):
    mod = pq.PQMF(100, 16).cuda()
    assert mod(torch.zeros(0, 1, 64, device="cuda")).shape == (0, 16, 4)
    assert mod(torch.zeros(2, 1, 0, device="cuda")).shape == (2, 16, 0)
    assert mod.inverse(torch.zeros(2, 16, 0, device="cuda")).shape == (2, 1, 0)
    y = mod(torch.ones(1, 1, 16, device="cuda"))
    assert y.shape == (1, 16, 1) and torch.isfinite(y).all()
    one = pq.PQMF(100, 1, polyphase=False) if False else None  # n_band == 1 is an identity in the reference
    with pytest.raises(RuntimeError):
        mod(torch.zeros(4, 64, device="cuda"))  # 2-D input
    with pytest.raises(RuntimeError):
        mod(torch.zeros(1, 1, 64))  # CPU tensor: no fallback
    with pytest.raises(RuntimeError):
        mod(torch.zeros(1, 1, 64, device="cuda", dtype=torch.float64))


# ------------------------------------------------------------------ size-independent properties at full size
def test_config2_properties_full_size(pq):
    """BASELINE config 2 (64 x 2^20): linearity, shift covariance by 2M, near-perfect reconstruction."""
    torch.manual_seed(0)
    mod = pq.PQMF(100, 16).cuda()
    b, t = 64, 1 << 20
    x = (0.5 * torch.randn(b, 1, t, device="cuda")).clamp_(-1, 1)
    y = mod(x)
    out = mod.inverse(y)
    err = out - x
    snr = 10 * torch.log10((x[..., 4096:-4096] ** 2).sum() / (err[..., 4096:-4096] ** 2).sum())
    assert snr.item() > 55.0  # interior SNR of the near-PR bank on noise (SURVEY section 6: ~60 dB)
    x2 = torch.roll(x, 32, dims=-1)
    y2 = mod(x2)
    assert (y2[..., 40:-40] - torch.roll(y, 2, dims=-1)[..., 40:-40]).abs().max().item() <= 2e-6
    a = mod(0.25 * x) - 0.25 * y
    assert a.abs().max().item() <= 2e-6
    # every batch row is processed independently and identically
    assert torch.equal(mod(x[5:6]), y[5:6])


# ------------------------------------------------------------------ the offline n_band 16 default (Hankel-4 kernels) vs the oracle
# These shapes have >= 96 tiles of 512 frames, so the dispatcher picks hankel4.cuh (smaller ones above run the fold kernels).
@pytest.mark.parametrize("b,frames", ((24, 2048), (100, 516), (97, 515), (7, 512 * 14 + 8)))
def test_hankel4_offline_vs_oracle(golden, pq, lib, b, frames):
    hk = golden("bank_M16.npz")["hk"]
    t = 16 * frames
    x = O.audio_like((b, 1, t), 99 + frames)
    mod = pq.PQMF(100, 16).cuda()
    assert (mod._flags >> 17) & 7 and (mod._flags >> 20) & 7  # the default bank allows trimmed correction steps
    y = mod(dev(x)).cpu().numpy()
    y64 = O.analysis(x[:, 0], hk)
    assert np.abs(y - y64).max() <= TOL / 2
    s = y64.astype(np.float32)
    out = mod.inverse(dev(s)).cpu().numpy()
    assert np.abs(out[:, 0] - O.synthesis(s, hk)).max() <= TOL / 2
    # the fold kernels (PQMF_FLAG_FOLD) and the Hankel-4 kernels are two implementations of the same arithmetic
    tables = mod._tables
    yf = torch.ops.pqmf_b200.analysis(dev(x), mod.hk, tables, frames, mod._flags | lib.PQMF_FLAG_FOLD)
    assert (yf.cpu().numpy() - y).__abs__().max() <= 3e-6
    of = torch.ops.pqmf_b200.synthesis(dev(s), mod.hk, tables, 0, mod._flags | lib.PQMF_FLAG_FOLD)
    assert (of.cpu().numpy() - out).__abs__().max() <= 6e-6


def test_hankel4_cached_offline_and_ragged(golden, pq):
    """CachedPQMF offline on the Hankel-4 path: ceil(T/M) frames, synthesis one frame later (o = 15: no alignment pad)."""
    hk = golden("bank_M16.npz")["hk"]
    b, t = 26, 16 * 2048 - 5
    x = O.audio_like((b, 1, t), 7)
    mod = pq.CachedPQMF(100, 16).cuda()
    y = mod(dev(x)).cpu().numpy()
    assert y.shape[-1] == 2048
    y64 = O.analysis(x[:, 0], hk, n_frames=2048)
    assert np.abs(y - y64).max() <= TOL / 2
    s = y64.astype(np.float32)
    out = mod.inverse(dev(s)).cpu().numpy()
    assert np.abs(out[:, 0] - O.synthesis(s, hk, delay_frames=1)).max() <= TOL / 2


def test_hankel4_worst_case_signals(golden, pq):
    """Inputs built to maximise what the trimmed correction steps drop: full-scale values whose signs follow the bank's
    tails (analysis) and all sixteen sub-bands at full scale with aligned signs (synthesis)."""
    hk = golden("bank_M16.npz")["hk"].astype(np.float64)
    b, frames = 24, 2048
    t = 16 * frames
    rng = np.random.default_rng(5)
    # analysis: x[n*16 + j - 256] = sign(hk[k, j]) for one band k per row, tiled along time with period 512 (a square-ish wave)
    x = np.empty((b, 1, t), np.float32)
    for r in range(b):
        pat = np.sign(hk[r % 16])
        pat[pat == 0] = 1.0
        x[r, 0] = np.tile(pat, t // 512 + 1)[:t] * (1.0 - 2.0 ** -12)  # not exactly representable in fp16
    mod = pq.PQMF(100, 16).cuda()
    y = mod(dev(x)).cpu().numpy()
    assert np.abs(y - O.analysis(x[:, 0].astype(np.float64), hk)).max() <= TOL
    # synthesis: every band at +-(1 - 2^-12) with random signs held for 32 frames
    s = (rng.integers(0, 2, (b, 16, frames // 32)) * 2 - 1).repeat(32, axis=2).astype(np.float32) * np.float32(1.0 - 2.0 ** -12)
    out = mod.inverse(dev(s)).cpu().numpy()
    ref = O.synthesis(s.astype(np.float64), hk)
    assert np.abs(out[:, 0] - ref).max() <= TOL * max(1.0, np.abs(ref).max())


@pytest.mark.parametrize("m", (32, 64))
def test_hankel4_worst_case_analysis_long_banks(pq, m):
    """n_band 32 / 64 trim 9 / 16 correction steps per side (their tails are long): full-scale inputs whose signs follow one band's taps,
    tiled with the bank's period -- what those steps drop adds up coherently -- stay within the tolerance of the fp64 closed form."""
    mod = pq.PQMF(100, m).cuda()
    trim_a = ((mod._flags >> 17) & 7) | (((mod._flags >> 24) & 3) << 3)
    assert trim_a > 7
    hk = mod.hk.cpu().numpy().astype(np.float64)
    L = hk.shape[1]
    b, frames = 24, 1024
    t = m * frames
    x = np.empty((b, 1, t), np.float32)
    for r in range(b):
        pat = np.sign(hk[(5 * r) % m])
        pat[pat == 0] = 1.0
        x[r, 0] = np.roll(np.tile(pat, t // L + 2), -(L // 2) + m * (r % 7))[:t] * (1.0 - 2.0 ** -12)
    y = mod(dev(x)).cpu().numpy()
    assert np.abs(y - O.analysis(x[:, 0].astype(np.float64), hk)).max() <= TOL


def test_hankel4_full_length_bank(golden, pq):
    """attenuation 120: the prototype no longer leaves 64 zero taps on each side, so the 512-tap instantiations run."""
    g = golden("bank_M16_att120.npz")
    hk = g["hk"]
    mod = pq.PQMF(120, 16).cuda()
    assert np.abs(mod.hk.cpu().numpy() - hk).max() <= 1e-7
    b, frames = 24, 2048
    x = O.audio_like((b, 1, 16 * frames), 120)
    y = mod(dev(x)).cpu().numpy()
    y64 = O.analysis(x[:, 0], hk)
    assert np.abs(y - y64).max() <= TOL / 2
    s = y64.astype(np.float32)
    out = mod.inverse(dev(s)).cpu().numpy()
    assert np.abs(out[:, 0] - O.synthesis(s, hk)).max() <= TOL / 2


# ------------------------------------------------------------------ n_band 8 / 32 on the 64-samples-per-row Hankel kernels
@pytest.mark.parametrize("m,b,frames", ((8, 24, 4096), (8, 50, 2100), (32, 24, 1024), (32, 49, 516), (8, 3, 8192 * 5 + 4), (4, 24, 8192), (4, 33, 6148),
                                         (4, 5, 2048 * 21 + 12)))
def test_hankel_other_band_counts_vs_oracle(golden, pq, m, b, frames):
    """>= 96 tiles of 8192 samples: the dispatcher picks hankel4.cuh for n_band 4, 8 and 32 too (same MMA shapes, N = 128)."""
    hk = golden(f"bank_M{m}.npz")["hk"]
    t = m * frames
    x = O.audio_like((b, 1, t), 7 * m + frames)
    mod = pq.PQMF(100, m).cuda()
    assert mod._tables.numel() > 0
    y = mod(dev(x)).cpu().numpy()
    y64 = O.analysis(x[:, 0], hk)
    assert np.abs(y - y64).max() <= TOL / 2
    s = y64.astype(np.float32)
    out = mod.inverse(dev(s)).cpu().numpy()
    assert np.abs(out[:, 0] - O.synthesis(s, hk)).max() <= TOL / 2
    # identical to the register-tiled direct form (exact=True) within the tolerance
    ex = pq.PQMF(100, m, exact=True).cuda()
    assert (ex(dev(x)).cpu().numpy() - y).__abs__().max() <= 3e-6
    # CachedPQMF: one frame later
    cached = pq.CachedPQMF(100, m).cuda()
    oc = cached.inverse(dev(s)).cpu().numpy()
    assert np.abs(oc[:, 0] - O.synthesis(s, hk, delay_frames=1)).max() <= TOL / 2


@pytest.mark.parametrize("att,m", ((60, 16), (140, 16), (60, 32), (140, 8), (60, 8), (80, 16), (100, 64), (120, 32), (60, 64), (80, 4), (120, 4)))
def test_hankel_other_prototype_lengths(pq, att, m):
    """Prototype lengths other than 32 n_band (L = 16 M or 64 M): tap span, K-steps and trims come from the actual bank.  Banks too
    long for one SM's shared memory (n_band 64; attenuation 120 at n_band 32) run as two tap ranges, the second launch accumulating."""
    mod = pq.PQMF(att, m).cuda()
    assert mod._tables.numel() > 0
    hk = mod.hk.cpu().numpy()
    b, t = 24, 32768
    x = O.audio_like((b, 1, t), att + m)
    tol = TOL / 2 if m < 64 else TOL  # at n_band 64 fp32 accumulation of 64 x 24 products with gain 64 alone is ~4e-6 (any fp32 path)
    y = mod(dev(x)).cpu().numpy()
    y64 = O.analysis(x[:, 0], hk)
    assert np.abs(y - y64).max() <= TOL / 2
    s = y64.astype(np.float32)
    out = mod.inverse(dev(s)).cpu().numpy()
    assert np.abs(out[:, 0] - O.synthesis(s, hk)).max() <= tol
    ex = pq.PQMF(att, m, exact=True).cuda()
    assert (ex(dev(x)).cpu().numpy() - y).__abs__().max() <= 3e-6
    cached = pq.CachedPQMF(att, m).cuda()
    oc = cached.inverse(dev(s)).cpu().numpy()
    assert np.abs(oc[:, 0] - O.synthesis(s, hk, delay_frames=1)).max() <= tol


@pytest.mark.parametrize("att,m,split", ((100, 64, True), (120, 32, True), (100, 32, False), (50, 64, False)))
def test_launch_count_counts_both_tap_ranges_of_split_banks(lib, pq, att, m, split):
    """pqmf_launch_count counts kernels: a split bank's two tap ranges are two launches per direction.  Its int16 synthesis stores
    through the direct form (the second range accumulates, not in int16): one launch."""
    mod = pq.PQMF(att, m).cuda()
    assert bool(mod._flags & lib.PQMF_FLAG_H4_SPLIT) == split
    hk, tab, L, fl = mod.hk.data_ptr(), mod._tables.data_ptr(), mod.hk.shape[1], mod._flags
    b, t = 32, 32768  # 128 tiles of 8192 samples: the offline Hankel-4 kernels
    f = t // m
    torch.manual_seed(att + m)
    x = (0.5 * torch.randn(b, t, device="cuda")).clamp_(-1, 1)
    pcm = (x * 32767).to(torch.int16)
    y = torch.empty(b, m, f, device="cuda")
    out = torch.empty(b, t, device="cuda")
    out16 = torch.empty(b, t, dtype=torch.int16, device="cuda")
    c, st = lib.cabi, torch.cuda.current_stream().cuda_stream
    calls = {
        "analysis": lambda: c.pqmf_analysis_f32(x.data_ptr(), y.data_ptr(), hk, tab, b, t, f, m, L, fl, st),
        "synthesis": lambda: c.pqmf_synthesis_f32(y.data_ptr(), out.data_ptr(), hk, tab, b, f, m, L, 0, fl, st),
        "pcm_analysis": lambda: c.pqmf_analysis_pcm16(pcm.data_ptr(), y.data_ptr(), hk, tab, b, t, 1, 0, f, m, L, fl, st),
        "pcm_synthesis": lambda: c.pqmf_synthesis_pcm16(y.data_ptr(), out16.data_ptr(), hk, tab, b, 1, f, m, L, 0, fl, st),
    }
    want = {"analysis": 2, "synthesis": 2, "pcm_analysis": 2, "pcm_synthesis": 1} if split else dict.fromkeys(calls, 1)
    got = {}
    for name, call in calls.items():
        n0 = lib.launch_count()
        rc = call()
        got[name] = (rc, lib.launch_count() - n0)
    torch.cuda.synchronize()
    assert got == {name: (0, n) for name, n in want.items()}


def test_cta_pair_and_single_cta_kernels_are_bit_identical(pq, lib):
    """PQMF_FLAG_NO_PAIR selects the one-CTA-per-SM launch of the same kernels: identical arithmetic, identical bits (odd tile
    counts exercise the pair's padding tile)."""
    mod = pq.PQMF(100, 16).cuda()
    torch.manual_seed(3)
    for b, frames in ((25, 2564), (97, 516), (1, 512 * 97)):
        x = (0.5 * torch.randn(b, 1, 16 * frames, device="cuda")).clamp_(-1, 1)
        y_pair = torch.ops.pqmf_b200.analysis(x, mod.hk, mod._tables, frames, mod._flags)
        y_one = torch.ops.pqmf_b200.analysis(x, mod.hk, mod._tables, frames, mod._flags | lib.PQMF_FLAG_NO_PAIR)
        assert torch.equal(y_pair, y_one)
        o_pair = torch.ops.pqmf_b200.synthesis(y_one, mod.hk, mod._tables, 0, mod._flags)
        o_one = torch.ops.pqmf_b200.synthesis(y_one, mod.hk, mod._tables, 0, mod._flags | lib.PQMF_FLAG_NO_PAIR)
        assert torch.equal(o_pair, o_one)


def test_custom_bank_that_is_not_window_times_cosine(golden, pq):
    """A hand-edited hk (loaded through the state dict) breaks the fold factorisation; the module then keeps the Hankel kernels,
    which take hk as it is, for both the streaming-size and the offline-batch paths."""
    hk = golden("bank_M16.npz")["hk"].copy()
    rng = np.random.default_rng(0)
    hk[:, 100:400] *= (1.0 + 0.05 * rng.standard_normal((16, 300))).astype(np.float32)
    mod = pq.PQMF(100, 16).cuda()
    sd = mod.state_dict()
    sd["hk"] = torch.from_numpy(hk)
    mod.load_state_dict(sd)
    assert mod.fold_residual > 1e-6 and mod._tables.numel() > 0
    for b, t in ((2, 16 * 600), (24, 32768)):
        x = O.audio_like((b, 1, t), 3 + b)
        y = mod(dev(x)).cpu().numpy()
        y64 = O.analysis(x[:, 0], hk)
        assert np.abs(y - y64).max() <= TOL / 2
        s = y64.astype(np.float32)
        out = mod.inverse(dev(s)).cpu().numpy()
        assert np.abs(out[:, 0] - O.synthesis(s, hk)).max() <= TOL / 2


@pytest.mark.parametrize("m,b,t", ((16, 64, 1 << 18), (16, 3, 16 * 1000), (8, 40, 8 * 8192), (32, 5, 32 * 300), (16, 200, 16 * 2048)))
def test_fused_process_equals_forward_then_inverse(pq, m, b, t):
    """process() = forward() then inverse() as one op (PQMFWrapper.process): the same bits, for every kernel path."""
    torch.manual_seed(m + b)
    x = (0.5 * torch.randn(b, 1, t, device="cuda")).clamp_(-1, 1)
    for cls, ragged in ((pq.PQMF, 0), (pq.CachedPQMF, 5)):
        mod = cls(100, m).cuda()
        xs = x[..., : t - ragged].contiguous() if ragged else x
        y = mod(xs)
        out = mod.inverse(y)
        out_f, y_f = mod.process(xs)
        assert torch.equal(y, y_f) and torch.equal(out, out_f)
        scripted = torch.jit.script(mod)
        out_s, y_s = scripted.process(xs)
        assert torch.equal(out_s, out) and torch.equal(y_s, y)
    xg = x[:2].clone().requires_grad_(True)
    out_g, _ = mod.process(xg)  # falls back to the differentiable ops
    out_g.square().sum().backward()
    assert xg.grad is not None and torch.isfinite(xg.grad).all()


@pytest.mark.parametrize("scale", (1e-3, 1.0, 300.0, 2.0e4))
def test_hankel_kernels_are_scale_covariant(golden, pq, scale):
    """The fp16 two-term split keeps relative accuracy up to the fp16 range (|x| < 65 504): errors scale with the signal.  Downwards
    there is an absolute floor instead: the second term of a sample below ~0.1 is an fp16 subnormal (step 6e-8), so quiet signals
    keep ~3e-8 per sample of absolute accuracy (-150 dBFS), not the relative accuracy of fp32."""
    hk = golden("bank_M16.npz")["hk"]
    b, t = 24, 32768
    x = (O.audio_like((b, 1, t), 77) * scale).astype(np.float32)
    mod = pq.PQMF(100, 16).cuda()
    y = mod(dev(x)).cpu().numpy()
    y64 = O.analysis(x[:, 0].astype(np.float64), hk)
    assert np.isfinite(y).all() and np.abs(y - y64).max() <= TOL / 2 * scale + 2e-7
    s = y64.astype(np.float32)
    out = mod.inverse(dev(s)).cpu().numpy()
    assert np.isfinite(out).all() and np.abs(out[:, 0] - O.synthesis(s.astype(np.float64), hk)).max() <= TOL / 2 * scale + 1e-6


def test_cuda_graph_capture_and_replay(pq):
    """The kernels (cluster launches with programmatic stream serialisation included) can be captured into a CUDA graph and replayed;
    the shared-memory opt-in happens on the warm-up call outside the capture."""
    mod = pq.PQMF(100, 16).cuda()
    torch.manual_seed(9)
    x = (0.5 * torch.randn(32, 1, 1 << 17, device="cuda")).clamp_(-1, 1)
    with torch.no_grad():
        ref = mod.inverse(mod(x))
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        s = torch.cuda.Stream()
        with torch.cuda.stream(s):
            mod.inverse(mod(x))
            s.synchronize()
            with torch.cuda.graph(g, stream=s):
                out = mod.inverse(mod(x))
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, ref)
        x.copy_(x.flip(0).contiguous())
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, mod.inverse(mod(x)))


@pytest.mark.parametrize("m,b,t", ((16, 64, 1 << 18), (16, 3, 16 * 1000), (8, 40, 8 * 8192), (32, 5, 32 * 300), (16, 200, 16 * 2048 - 7)))
def test_reconstruct_without_subbands_equals_process(pq, m, b, t):
    """reconstruct() = inverse(forward(x)) with the sub-bands in an L2-sized scratch instead of a tensor (the Pvoc wrapper's forward,
    1-PitchShifterWrapper.py:303-316): the same bits as process()'s reconstruction, for every kernel path and for ragged cached lengths."""
    torch.manual_seed(m + b)
    x = (0.5 * torch.randn(b, 1, t, device="cuda")).clamp_(-1, 1)
    for cls in (pq.PQMF, pq.CachedPQMF):
        if cls is pq.PQMF and t % m:
            continue
        mod = cls(100, m).cuda()
        want, _ = mod.process(x)
        assert torch.equal(mod.reconstruct(x), want)
        assert torch.equal(torch.jit.script(mod).reconstruct(x), want)
    xg = x[:2].clone().requires_grad_(True)
    mod.reconstruct(xg).square().sum().backward()
    assert xg.grad is not None and torch.isfinite(xg.grad).all()


@pytest.mark.parametrize("scale,tol", ((1e-6, 2e-10), (1e-4, 5e-10), (1e-3, 5e-9), (1.0, 5e-6), (2.0e4, 0.1)))
def test_quiet_and_loud_signals_keep_relative_accuracy(golden, pq, scale, tol):
    """Round 2: the second fp16 term is scaled by 2^11, so the tensor-core kernels keep RELATIVE accuracy (TOL / 2 of the signal scale)
    down to 1e-4 of full scale, and an absolute floor of ~1e-11 per sample below that (it was 3e-8); check_range=True routes anything
    beyond to plain fp32."""
    hk = golden("bank_M16.npz")["hk"]
    b, t = 24, 32768
    x = (O.audio_like((b, 1, t), 78) * scale).astype(np.float32)
    mod = pq.PQMF(100, 16).cuda()
    y = mod(dev(x)).cpu().numpy()
    y64 = O.analysis(x[:, 0].astype(np.float64), hk)
    assert np.isfinite(y).all() and np.abs(y - y64).max() <= tol
    s = y64.astype(np.float32)
    out = mod.inverse(dev(s)).cpu().numpy()
    assert np.isfinite(out).all() and np.abs(out[:, 0] - O.synthesis(s.astype(np.float64), hk)).max() <= 2 * tol


def test_check_range_routes_out_of_range_inputs_to_fp32(golden, pq):
    hk = golden("bank_M16.npz")["hk"]
    x = (O.audio_like((24, 1, 32768), 79) * 1.0e5).astype(np.float32)   # beyond the fp16 range of the tensor-core kernels
    guarded = pq.PQMF(100, 16, check_range=True).cuda()
    y = guarded(dev(x)).cpu().numpy()
    y64 = O.analysis(x[:, 0].astype(np.float64), hk)
    assert np.isfinite(y).all() and np.abs(y - y64).max() <= 1e-5 * 1.0e5
    plain = pq.PQMF(100, 16, fp32=True).cuda()
    assert np.array_equal(plain(dev(x)).cpu().numpy(), y)
    tiny = (O.audio_like((24, 1, 32768), 80) * 1.0e-9).astype(np.float32)
    yt = guarded(dev(tiny)).cpu().numpy()
    assert np.abs(yt - O.analysis(tiny[:, 0].astype(np.float64), hk)).max() <= 1e-5 * 1.0e-9
    assert torch.jit.script(guarded)(dev(x)).shape == (24, 16, 2048)
