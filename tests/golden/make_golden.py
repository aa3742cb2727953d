"""Regenerates tests/golden/*.npz by running the REFERENCE ITSELF in the dev container.

    python tests/golden/make_golden.py            # needs /root/reference (read-only mount)

The reference (`/root/reference/pqmf.py`) is imported unmodified; the only thing added
is an in-memory stand-in for the third-party `cached_conv` package it imports at module
top (pqmf.py:3), which is neither vendored nor installed.  The stand-in implements the
*non-cached* `cached_conv.Conv1d` exactly as it is baked into the reference's committed
TorchScript archive PitchShifterPvoc/torchscript/pqmfpvoc.ts
(code/__torch__/cached_conv/convs.py: `F.pad(x, self._pad)` then `conv1d`), and the
archive itself is loaded as a second, shim-free oracle for the offline CachedPQMF path.

/root/reference does not exist on the GPU box, so nothing else in the repo reads it at
test/bench time: the vectors written here are what travels.
"""
from __future__ import annotations

import hashlib
import os
import sys
import types
import wave

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

REF = os.environ.get("PQMF_REFERENCE", "/root/reference")
OUT = os.path.dirname(os.path.abspath(__file__))


def install_cached_conv_stand_in():
    cc = types.ModuleType("cached_conv")

    def get_padding(kernel_size, stride=1, dilation=1, mode="centered"):
        if kernel_size == 1:
            return (0, 0)
        p = (kernel_size - 1) * dilation + 1
        return (p // 2, p // 2)

    class Conv1d(nn.Conv1d):
        def __init__(self, *args, **kwargs):
            self._pad = kwargs.get("padding", (0, 0))
            kwargs["padding"] = 0
            super().__init__(*args, **kwargs)
            self.cumulative_delay = 0

        def script_cache(self):
            pass

        def forward(self, x):
            return F.conv1d(F.pad(x, self._pad), self.weight, self.bias, self.stride, 0, self.dilation, self.groups)

    cc.get_padding = get_padding
    cc.Conv1d = Conv1d
    sys.modules["cached_conv"] = cc


def read_pcm16(path):
    with wave.open(path, "rb") as w:
        assert w.getsampwidth() == 2
        n_ch, sr, n = w.getnchannels(), w.getframerate(), w.getnframes()
        pcm = np.frombuffer(w.readframes(n), dtype="<i2").reshape(n, n_ch).T.copy()
    return pcm, sr


def audio_like(shape, seed):
    rng = np.random.default_rng(seed)
    return np.clip(0.5 * rng.standard_normal(shape), -1.0, 1.0).astype(np.float32)


def snr_db(ref, est):
    ref = ref.astype(np.float64)
    est = est.astype(np.float64)
    return float(10 * np.log10(np.sum(ref ** 2) / np.sum((ref - est) ** 2)))


def main():
    install_cached_conv_stand_in()
    sys.path.insert(0, REF)
    import pqmf as ref  # the reference, unmodified

    torch.manual_seed(0)
    torch.set_grad_enabled(False)
    meta = {"torch": torch.__version__, "numpy": np.__version__}
    import scipy

    meta["scipy"] = scipy.__version__
    # CPU conv1d bits also depend on these: tests/test_oracle.py reproduces the thread count and checks the level
    meta["cpu_capability"] = torch.backends.cpu.get_cpu_capability()
    meta["threads"] = torch.get_num_threads()

    # ---- banks: h, hk for every n_band the configs name (attenuation 100) + attenuation sweep at M=16
    for m in (2, 4, 8, 16, 32, 64):
        p = ref.PQMF(100, m)
        np.savez_compressed(os.path.join(OUT, f"bank_M{m}.npz"), h=p.h.numpy(), hk=p.hk.numpy(),
                            h_sha256=hashlib.sha256(p.h.numpy().tobytes()).hexdigest())
    for att in (80, 120):
        p = ref.PQMF(att, 16)
        np.savez_compressed(os.path.join(OUT, f"bank_M16_att{att}.npz"), h=p.h.numpy(), hk=p.hk.numpy())
    p12 = ref.PQMF(100, 12, polyphase=False)  # non power of two: classic only (pqmf.py:220-224)
    np.savez_compressed(os.path.join(OUT, "bank_M12_classic.npz"), h=p12.h.numpy(), hk=p12.hk.numpy())

    # ---- the committed TorchScript archive (offline CachedPQMF, M=16)
    ts = torch.jit.load(os.path.join(REF, "PitchShifterPvoc/torchscript/pqmfpvoc.ts")).pqmf
    x_ts = torch.from_numpy(audio_like((2, 1, 4096), 77))
    y_ts = ts.forward(x_ts)
    o_ts = ts.inverse(y_ts)
    np.savez_compressed(os.path.join(OUT, "ts_M16.npz"), h=ts.h.numpy(), hk=ts.hk.numpy(),
                        fwd_weight_shape=np.array(ts.forward_conv.weight.shape), fwd_pad=np.array(ts.forward_conv._pad),
                        inv_weight=ts.inverse_conv.weight.detach().numpy(), inv_pad=np.array(ts.inverse_conv._pad),
                        x=x_ts.numpy(), y=y_ts.numpy(), out=o_ts.numpy())

    # ---- per-n_band vectors: polyphase / classic / cached, fp32 reference outputs
    for m in (4, 8, 16, 32, 64):
        pp = ref.PQMF(100, m, polyphase=True)
        pc = ref.PQMF(100, m, polyphase=False)
        cp = ref.CachedPQMF(100, m)
        length = pp.hk.shape[1]
        t = 4 * length
        x = torch.from_numpy(audio_like((2, 1, t), 1000 + m))
        y_poly = pp.forward(x)
        y_classic = pc.forward(x)
        y_cached = cp.forward(x)
        out_poly = pp.inverse(y_poly)
        out_classic = pc.inverse(y_poly)
        out_cached = cp.inverse(y_poly)
        # ragged length (T % M != 0): classic -> floor(T/M) frames, cached -> ceil(T/M) frames
        xr = x[..., : t - m // 2 - 1].contiguous()
        yr_classic = pc.forward(xr)
        yr_cached = cp.forward(xr)
        # unit-variance sub-bands (stress for synthesis; direct-form kernels must still meet 1e-5)
        s_rand = torch.randn(2, m, 64, generator=torch.Generator().manual_seed(2000 + m))
        out_rand = pp.inverse(s_rand)
        np.savez_compressed(
            os.path.join(OUT, f"vectors_M{m}.npz"), x=x.numpy(), y_poly=y_poly.numpy(), y_classic=y_classic.numpy(),
            y_cached=y_cached.numpy(), out_poly=out_poly.numpy(), out_classic=out_classic.numpy(),
            out_cached=out_cached.numpy(), x_ragged_len=np.array(xr.shape[-1]), yr_classic=yr_classic.numpy(),
            yr_cached=yr_cached.numpy(), s_rand=s_rand.numpy(), out_rand=out_rand.numpy())
    pc12 = p12
    x12 = torch.from_numpy(audio_like((1, 1, 12 * 100), 1012))
    y12 = pc12.forward(x12)
    np.savez_compressed(os.path.join(OUT, "vectors_M12_classic.npz"), x=x12.numpy(), y=y12.numpy(), out=pc12.inverse(y12).numpy())

    # ---- config 1: audio/flute.wav, padded to a multiple of 8192 as the wrappers do (PQMFWrapper.py:117-121)
    flute, sr = read_pcm16(os.path.join(REF, "audio/flute.wav"))
    violin, _ = read_pcm16(os.path.join(REF, "audio/violin_bow_nonvib_f4_44100.wav"))
    multi, sr_m = read_pcm16(os.path.join(REF, "audio/flutemulti.wav"))
    rows = {}
    for name, pcm in (("flute", flute), ("violin", violin)):
        n = pcm.shape[1]
        n_pad = -(-n // 8192) * 8192
        xf = np.zeros((1, 1, n_pad), np.float32)
        xf[0, 0, :n] = pcm[0].astype(np.float32) / 32768.0
        rows[name] = xf
    snr = {}
    for m in (2, 4, 8, 16, 32, 64):
        p = ref.PQMF(100, m)
        for name, xf in rows.items():
            xt = torch.from_numpy(xf)
            snr[f"{name}_M{m}"] = snr_db(xf, p.inverse(p.forward(xt)).numpy())
    p16 = ref.PQMF(100, 16)
    c16 = ref.CachedPQMF(100, 16)
    xt = torch.from_numpy(rows["flute"])
    y = p16.forward(xt)
    o = p16.inverse(y)
    oc = c16.inverse(c16.forward(xt))
    snr["flute_M16_cached_delay16"] = snr_db(rows["flute"][..., :-16], oc.numpy()[..., 16:])
    lo, hi = 131072, 131072 + 16384  # excerpt kept in full precision; the whole clip is pinned through the SNR + checksums
    np.savez_compressed(
        os.path.join(OUT, "flute_C1.npz"), pcm=flute[0], sr=np.array(sr), n_pad=np.array(xt.shape[-1]),
        y_excerpt=y.numpy()[:, :, lo // 16 : hi // 16], out_excerpt=o.numpy()[:, :, lo:hi], excerpt=np.array([lo, hi]),
        y_abs_max=np.array(np.abs(y.numpy()).max()), y_sum=np.array(y.numpy().astype(np.float64).sum()),
        out_sum=np.array(o.numpy().astype(np.float64).sum()),
        y_head=y.numpy()[:, :, :64], out_head=o.numpy()[:, :, :1024], out_tail=o.numpy()[:, :, -1024:],
        **{k: np.array(v) for k, v in snr.items()})
    # a short 2-channel excerpt of flutemulti.wav (config 4 folds channels into batch)
    np.savez_compressed(os.path.join(OUT, "flutemulti_excerpt.npz"), pcm=multi[:, 44100 : 44100 + 32768], sr=np.array(sr_m))
    with open(os.path.join(OUT, "VERSIONS.txt"), "w") as f:
        for k, v in meta.items():
            f.write(f"{k} {v}\n")
    for k, v in sorted(snr.items()):
        print(k, round(v, 3))


if __name__ == "__main__":
    main()
