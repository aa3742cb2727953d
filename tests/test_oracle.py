"""Pins the oracle (oracle/) against vectors produced by the reference itself
(tests/golden/make_golden.py).  CPU only."""
import hashlib
import os

import numpy as np
import pytest
import torch

from oracle import pqmf_oracle as O
from oracle import pqmf_port_torch as P

BANDS = (4, 8, 16, 32, 64)
# the reference's own fp32 run sits <= ~2e-6 from the float64 closed form (SURVEY.md fact 6)
FP64_VS_REF_FWD = 2e-6
FP64_VS_REF_INV = 6e-6


@pytest.mark.parametrize("m", (2, 4, 8, 16, 32, 64))
def test_design_reproduces_reference_bank(golden, m):
    g = golden(f"bank_M{m}.npz")
    h, hk = O.design_bank(100, m)
    assert h.dtype == np.float32 and hk.dtype == np.float32
    assert hashlib.sha256(h.tobytes()).hexdigest() == str(g["h_sha256"])  # bit for bit (SURVEY A.5)
    assert hk.shape == g["hk"].shape
    assert np.abs(hk - g["hk"]).max() <= 1e-8


def test_design_matches_committed_torchscript_archive(golden):
    g = golden("ts_M16.npz")
    h, hk = O.design_bank(100, 16)
    assert np.array_equal(h, g["h"])
    assert np.abs(hk - g["hk"]).max() <= 1e-8
    assert tuple(g["fwd_weight_shape"]) == (16, 1, 513) and tuple(g["fwd_pad"]) == (256, 256)
    assert g["inv_weight"].shape == (16, 16, 33) and tuple(g["inv_pad"]) == (16, 16)


@pytest.mark.parametrize("att", (80, 120))
def test_design_attenuation_sweep(golden, att):
    g = golden(f"bank_M16_att{att}.npz")
    h, hk = O.design_bank(att, 16)
    assert np.array_equal(h, g["h"]) and np.abs(hk - g["hk"]).max() <= 1e-8


@pytest.mark.parametrize("m", BANDS)
def test_closed_form_analysis_vs_reference(golden, m):
    g = golden(f"vectors_M{m}.npz")
    hk = golden(f"bank_M{m}.npz")["hk"]
    x = g["x"][:, 0]
    y = O.analysis(x, hk)
    for key in ("y_poly", "y_classic", "y_cached"):
        assert np.abs(y - g[key]).max() <= FP64_VS_REF_FWD, key
    # ragged T: classic -> floor(T/M) frames, cached -> ceil(T/M)
    tr = int(g["x_ragged_len"])
    xr = x[:, :tr]
    assert g["yr_classic"].shape[-1] == tr // m and g["yr_cached"].shape[-1] == -(-tr // m)
    assert np.abs(O.analysis(xr, hk, tr // m) - g["yr_classic"]).max() <= FP64_VS_REF_FWD
    assert np.abs(O.analysis(xr, hk, -(-tr // m)) - g["yr_cached"]).max() <= FP64_VS_REF_FWD


@pytest.mark.parametrize("m", BANDS)
def test_closed_form_synthesis_vs_reference(golden, m):
    g = golden(f"vectors_M{m}.npz")
    hk = golden(f"bank_M{m}.npz")["hk"]
    s = g["y_poly"]
    out = O.synthesis(s, hk)
    assert np.abs(out - g["out_poly"][:, 0]).max() <= FP64_VS_REF_INV
    assert np.abs(out - g["out_classic"][:, 0]).max() <= 2 * FP64_VS_REF_INV
    out_c = O.synthesis(s, hk, delay_frames=1)
    assert np.abs(out_c - g["out_cached"][:, 0]).max() <= FP64_VS_REF_INV
    # cached == offline delayed by exactly one frame (SURVEY fact 5)
    assert np.abs(out_c[:, m:] - out[:, :-m]).max() <= 1e-12
    out_r = O.synthesis(g["s_rand"], hk)
    assert np.abs(out_r - g["out_rand"][:, 0]).max() <= 4 * FP64_VS_REF_INV


def test_non_power_of_two_classic(golden):
    g = golden("vectors_M12_classic.npz")
    b = golden("bank_M12_classic.npz")
    h, hk = O.design_bank(100, 12)
    assert np.array_equal(h, b["h"]) and np.abs(hk - b["hk"]).max() <= 1e-8
    x = g["x"][:, 0]
    # L % M != 0 here: classic analysis is still the stride-M correlation
    y = O.analysis(x, hk, x.shape[1] // 12)
    assert np.abs(y - g["y"]).max() <= FP64_VS_REF_FWD


def test_torchscript_archive_outputs(golden):
    g = golden("ts_M16.npz")
    hk = g["hk"]
    y = O.analysis(g["x"][:, 0], hk)
    assert np.abs(y - g["y"]).max() <= FP64_VS_REF_FWD
    out = O.synthesis(g["y"], hk, delay_frames=1)
    assert np.abs(out - g["out"][:, 0]).max() <= FP64_VS_REF_INV


@pytest.fixture
def golden_env():
    """The environment tests/golden/VERSIONS.txt records for the vectors, with torch's CPU thread count set to the one they were
    made with for the duration of the test."""
    with open(os.path.join(os.path.dirname(__file__), "golden", "VERSIONS.txt")) as f:
        made_with = dict(line.split(" ", 1) for line in f.read().splitlines() if line)
    before = torch.get_num_threads()
    torch.set_num_threads(int(made_with.get("threads", before)))
    yield made_with
    torch.set_num_threads(before)


@pytest.mark.parametrize("m", BANDS)
def test_torch_port_is_bit_exact_with_reference(golden, golden_env, m):
    """Same op sequence, same torch build -> identical bits (when the golden file was made with this torch).  CPU conv1d also rounds
    differently at another instruction-set level of its kernels or another split over threads: the split is pinned by the fixture,
    and a host whose kernels run at another level gets the fp32-vs-fp32 bound instead of identical bits."""
    g = golden(f"vectors_M{m}.npz")
    hk = torch.from_numpy(golden(f"bank_M{m}.npz")["hk"])
    x = torch.from_numpy(g["x"])
    exact = golden_env.get("torch") == torch.__version__ and golden_env.get("cpu_capability") == torch.backends.cpu.get_cpu_capability()
    tol = 0.0 if exact else 2e-6

    def close(a, b, scale=1.0):
        return np.abs(a.numpy() - b).max() <= tol * scale

    y = P.analysis_polyphase(x, hk)
    assert close(y, g["y_poly"])
    assert close(P.analysis_classic(x, hk), g["y_classic"])
    assert close(P.analysis_cached_offline(x, hk), g["y_cached"])
    s = torch.from_numpy(g["y_poly"])
    assert close(P.synthesis_polyphase(s, hk), g["out_poly"], 4)
    assert close(P.synthesis_cached_offline(s, hk), g["out_cached"], 4)
    if m <= 16:  # zero-stuffed classic synthesis is very slow for large M
        assert close(P.synthesis_classic(s, hk), g["out_classic"], 4)


def test_flute_config1(golden):
    g = golden("flute_C1.npz")
    hk = golden("bank_M16.npz")["hk"]
    n_pad = int(g["n_pad"])
    x = np.zeros((1, n_pad), np.float32)
    x[0, : g["pcm"].shape[0]] = g["pcm"].astype(np.float32) / 32768.0
    y = O.analysis(x, hk)
    lo, hi = g["excerpt"]
    assert np.abs(y[:, :, lo // 16 : hi // 16] - g["y_excerpt"]).max() <= FP64_VS_REF_FWD
    assert np.abs(y[:, :, :64] - g["y_head"]).max() <= FP64_VS_REF_FWD
    assert abs(y.sum() - float(g["y_sum"])) <= 1e-3
    out = O.synthesis(y.astype(np.float32), hk)
    assert np.abs(out[:, lo:hi] - g["out_excerpt"][:, 0]).max() <= FP64_VS_REF_INV
    assert np.abs(out[:, :1024] - g["out_head"][:, 0]).max() <= FP64_VS_REF_INV
    assert np.abs(out[:, -1024:] - g["out_tail"][:, 0]).max() <= FP64_VS_REF_INV
    assert abs(O.snr_db(x, out) - float(g["flute_M16"])) <= 0.1  # 65.145 dB (SURVEY A.5)
    out_c = O.synthesis(y.astype(np.float32), hk, delay_frames=1)
    assert abs(O.snr_db(x[:, :-16], out_c[:, 16:]) - float(g["flute_M16_cached_delay16"])) <= 0.1


@pytest.mark.parametrize("m", (4, 16, 64))
def test_impulse_reads_bank_columns(golden, m):
    """SURVEY A.2: x = delta[t - t0]  =>  y[k, n] = sigma(k, n) * hk[k, t0 - n M + L/2]."""
    hk = golden(f"bank_M{m}.npz")["hk"].astype(np.float64)
    length = hk.shape[1]
    t = 4 * length
    t0 = length + 3
    x = np.zeros((1, t))
    x[0, t0] = 1.0
    y = O.analysis(x, hk)[0]
    sig = O.sign_mask(m, t // m)
    for n in range(t // m):
        j = t0 - n * m + length // 2
        col = hk[:, j] if 0 <= j < length else np.zeros(m)
        assert np.allclose(y[:, n], sig[:, n] * col, atol=0)


def test_shift_covariance_two_frames(golden):
    hk = golden("bank_M16.npz")["hk"]
    x = O.audio_like((1, 4096), 5).astype(np.float64)
    xs = np.concatenate([np.zeros((1, 32)), x[:, :-32]], axis=1)
    y, ys = O.analysis(x, hk), O.analysis(xs, hk)
    # (the last L/2M + 2 frames see the samples that the shift pushed out of the clip)
    assert np.abs(ys[:, :, 2:-20] - y[:, :, :-22]).max() <= 1e-12


@pytest.mark.parametrize("m,block", ((16, 2048), (16, 512), (8, 256), (64, 4096)))
def test_streaming_equals_offline_with_fixed_latency(golden, m, block):
    """SURVEY A.4 whole-signal invariants (exact in float64):
    stream_analysis(x)  == offline_cached_forward(cat[zeros(L/2), x])[..., :T/M]
    stream_synthesis(s) == offline_cached_inverse(cat[zeros(K/2 frames), s])[..., :T]"""
    hk = golden(f"bank_M{m}.npz")["hk"]
    length = hk.shape[1]
    k_taps = length // m
    n_blocks = 6
    t = n_blocks * block
    x = O.audio_like((3, t), 11).astype(np.float64)
    st = O.StreamState(3, m, length)
    ys, outs = [], []
    for i in range(n_blocks):
        yb = O.stream_analysis(x[:, i * block : (i + 1) * block], hk, st)
        ys.append(yb)
        outs.append(O.stream_synthesis(yb, hk, st))
    y_stream = np.concatenate(ys, axis=2)
    out_stream = np.concatenate(outs, axis=1)
    y_off = O.analysis(np.concatenate([np.zeros((3, length // 2)), x], axis=1), hk)[:, :, : t // m]
    assert np.abs(y_stream - y_off).max() <= 1e-13
    s_pad = np.concatenate([np.zeros((3, m, k_taps // 2)), y_stream], axis=2)
    out_off = O.synthesis(s_pad, hk, delay_frames=1)[:, :t]
    assert np.abs(out_stream - out_off).max() <= 1e-12
    # end-to-end latency L/2 + (K/2) M + M samples (528 at M=16), near-perfect reconstruction after it
    lat = length // 2 + (k_taps // 2) * m + m
    assert O.snr_db(x[:, : t - lat], out_stream[:, lat:]) > 30.0
