"""The reference's own wrapper scripts, UNCHANGED, running on CUDA on top of the drop-in (north_star: "usable unchanged by
PQMFWrapper.py and both pitch-shifter wrappers").  The wrapper files come, verbatim, out of the archive that
oracle/fetch_ref_wrappers.py packs where /root/reference is mounted (oracle/_ref/wrappers.tar: git-ignored, travels to the GPU box) and
are unpacked into a temporary directory here; the expected outputs in tests/golden/wrappers.npz were produced by the same files on top
of the REFERENCE's pqmf.py (tests/golden/make_golden_wrappers.py).  The wrapper scripts are not part of this repository, so the
PQMF stages they run are also checked against those stored outputs without them (test_dropin_stages_match_the_stored_wrapper_outputs)."""
import importlib.util
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARCHIVE = os.path.join(ROOT, "oracle", "_ref", "wrappers.tar")
pytestmark = pytest.mark.gpu
needs_wrapper_scripts = pytest.mark.skipif(
    not os.path.isfile(ARCHIVE), reason="oracle/_ref/wrappers.tar missing: pack the original project's wrapper scripts with oracle/fetch_ref_wrappers.py")
TOL = 1e-5
WRAPPERS = ""  # set by the fixture: where the archive was unpacked


def _load(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


@pytest.fixture(scope="module")
def dropin_on_path(tmp_path_factory):
    """`from pqmf import CachedPQMF` and `from PQMF.pqmf import CachedPQMF` resolve to the drop-in; the vocoder the Pvoc wrapper imports
    as PQMF.PitchShifterPvoc.VocoderPitchShifter resolves to the reference's own file."""
    global WRAPPERS
    sys.path.insert(0, ROOT)
    from oracle import fetch_ref_wrappers

    WRAPPERS = str(tmp_path_factory.mktemp("ref_wrappers"))
    assert fetch_ref_wrappers.unpack(WRAPPERS)
    del sys.path[0]
    sys.path[:0] = [os.path.join(ROOT, "dropin"), ROOT]
    for name in ("pqmf", "PQMF", "PQMF.pqmf"):
        sys.modules.pop(name, None)
    import PQMF
    import PQMF.pqmf
    import pqmf

    assert "pqmf_b200" in pqmf.CachedPQMF.__module__ and "pqmf_b200" in PQMF.pqmf.CachedPQMF.__module__
    PQMF.__path__.append(os.path.join(WRAPPERS, "PQMF"))
    yield
    PQMF.__path__.pop()
    del sys.path[:2]


@needs_wrapper_scripts
def test_pqmfwrapper_scripted_process_on_cuda(golden, dropin_on_path, tmp_path):
    g = golden("wrappers.npz")
    W = _load("PQMFWrapper", os.path.join(WRAPPERS, "PQMFWrapper.py"))
    w = W.PQMFWrapper(attenuation=100, n_band=16, m_buffer_size=8192).eval().cuda()
    x = torch.from_numpy(g["x"]).cuda()
    with torch.no_grad():
        recon, sub = w.process(x)                                # eager
        scripted = torch.jit.script(w)                           # what the reference exports (PQMFWrapper.py:102-108)
        path = str(tmp_path / "pqmf.ts")
        scripted.save(path)
        loaded = torch.jit.load(path)
        recon_s, sub_s = loaded.process(x)
    assert loaded.get_methods() == ["forward", "inverse", "process"]
    assert torch.equal(recon, recon_s) and torch.equal(sub, sub_s)
    assert np.abs(sub.cpu().numpy() - g["process_sub"]).max() <= TOL
    assert np.abs(recon.cpu().numpy() - g["process_recon"]).max() <= TOL
    with pytest.raises(ValueError):
        w.forward(torch.zeros(2, 3, 64, device="cuda"))          # the wrapper's own shape check still fires


@needs_wrapper_scripts
def test_pvoc_pitch_shifter_wrapper_on_cuda(golden, dropin_on_path):
    g = golden("wrappers.npz")
    P = _load("pvoc_wrapper", os.path.join(WRAPPERS, "PQMF", "PitchShifterPvoc", "1-PitchShifterWrapper.py"))
    w = P.PQMFPitchShiftWrapper(attenuation=100, n_band=16, m_buffer_size=8192, sample_rate=44100).eval().cuda()
    x = torch.from_numpy(g["x"]).cuda()
    with torch.no_grad():
        y = w.forward(x[:, :8192])                               # PQMF stages only (1-PitchShifterWrapper.py:303-316)
        p0 = w.pitchshift(x[:, :8192])                           # decompose -> 16 phase vocoders -> cross-fade -> crop/pad -> cat -> inverse
        p1 = w.pitchshift(x[:, 8192:])
    assert np.abs(y.cpu().numpy() - g["pvoc_forward"]).max() <= TOL
    # the vocoders in between (STFT / phase arithmetic in fp32 on a different device) are not ours: same signal to their own rounding
    for ours, key in ((p0, "pvoc_pitch_block0"), (p1, "pvoc_pitch_block1")):
        ref = g[key]
        assert ours.shape == ref.shape and torch.isfinite(ours).all()
        assert np.abs(ours.cpu().numpy() - ref).max() <= 2e-3 * max(1.0, float(np.abs(ref).max()))
    scripted = torch.jit.script(w)                               # the reference exports this wrapper too (:337-343)
    with torch.no_grad():
        assert torch.equal(scripted.forward(x[:, :8192]), y)


@needs_wrapper_scripts
def test_torchaudio_pitch_shifter_wrapper_on_cuda(golden, dropin_on_path):
    g = golden("wrappers.npz")
    T = _load("ps_wrapper", os.path.join(WRAPPERS, "PQMF", "PitchShifterTorchaudio", "PQMFPsWrapper.py"))
    w = T.PQMFPitchShiftWrapper(attenuation=100, n_band=16, m_buffer_size=512, sample_rate=44100).eval().cuda()
    x = torch.from_numpy(g["x"]).cuda()
    with torch.no_grad():
        sub = w.forward(x[:, :8192])
        rec = w.inverse(sub)
        shifted = w.pitchshifter(x[:, :8192])
    assert np.abs(sub.cpu().numpy() - g["ps_forward"]).max() <= TOL
    assert np.abs(rec.cpu().numpy() - g["ps_inverse"]).max() <= TOL
    ref = g["ps_pitch"]
    assert shifted.shape == ref.shape and torch.isfinite(shifted).all()
    assert np.abs(shifted.cpu().numpy() - ref).max() <= 2e-3 * max(1.0, float(np.abs(ref).max()))


def test_dropin_stages_match_the_stored_wrapper_outputs(golden):
    """The PQMF stages of the three wrappers -- CachedPQMF(100, 16) forward and inverse on a [1, 1, T] block, fresh module, no stream
    state -- against what the original wrappers returned on top of the original pqmf.py (wrappers.npz), without the wrapper scripts."""
    import pqmf_b200 as pq

    g = golden("wrappers.npz")
    mod = pq.CachedPQMF(attenuation=100, n_band=16).eval().cuda()
    x = torch.from_numpy(g["x"]).cuda()[None]                     # the wrappers' own unsqueeze(0) of their [1, T] input
    with torch.no_grad():
        sub = mod(x)                                             # PQMFWrapper.process
        recon = mod.inverse(sub)
        sub_b = mod(x[..., :8192].contiguous())                  # PQMFPsWrapper.forward / .inverse on the first block
        rec_b = mod.inverse(sub_b)
    assert np.abs(sub.cpu().numpy() - g["process_sub"]).max() <= TOL
    assert np.abs(recon.cpu().numpy() - g["process_recon"]).max() <= TOL
    assert np.abs(sub_b.cpu().numpy() - g["ps_forward"]).max() <= TOL
    assert np.abs(rec_b.cpu().numpy() - g["ps_inverse"]).max() <= TOL
    assert np.abs(rec_b[0].cpu().numpy() - g["pvoc_forward"]).max() <= TOL   # the Pvoc wrapper's forward: reconstruction, [1, T]
