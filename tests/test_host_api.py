"""CPU-side checks: the C-ABI library loads and exports every symbol include/pqmf_b200.h declares, the
module API mirrors the reference's (constructor, buffers, state_dict keys, errors, TorchScript), and nothing
falls back to the CPU."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def pq():
    import pqmf_b200

    return pqmf_b200


def test_cabi_exports_every_declared_symbol(pq):
    header = open(os.path.join(ROOT, "include", "pqmf_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(pqmf_[a-z0-9_]+)\s*\(", header))
    assert {"pqmf_analysis_f32", "pqmf_synthesis_f32", "pqmf_analysis_stream_f32", "pqmf_synthesis_stream_f32",
            "pqmf_build_tables_f32", "pqmf_roundtrip_host_f32", "pqmf_analysis_pcm16", "pqmf_synthesis_pcm16", "pqmf_synthesis_bands_f32",
            "pqmf_reconstruct_f32", "pqmf_roundtrip_host_pcm16", "pqmf_roundtrip_host_multi_f32"} <= declared
    lib = ctypes.CDLL(pq.library_paths()[0])
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/pqmf_b200.h but not exported"
    assert lib.pqmf_abi_version() == 2


def test_torch_ops_are_registered_for_cuda_only(pq):
    for op in ("analysis", "synthesis", "analysis_stream", "synthesis_stream"):
        assert hasattr(torch.ops.pqmf_b200, op)
    mod = pq.PQMF(100, 16)
    with pytest.raises((RuntimeError, NotImplementedError)) as e:
        mod(torch.zeros(1, 1, 64))
    assert "CPU" in str(e.value)  # no CPU fallback: the dispatcher has no CPU kernel for the op


def test_module_surface_matches_reference(pq, golden):
    mod = pq.CachedPQMF(100, 16)
    assert list(mod.state_dict().keys()) == ["hk", "h", "forward_conv.weight", "inverse_conv.weight"]
    assert mod.n_band == 16 and mod.polyphase is True and mod.n_channels == 1
    assert mod.hk.shape == (16, 512) and mod.h.shape == (377,)
    assert mod.forward_conv.weight.shape == (16, 1, 513) and mod.forward_conv._pad == (256, 256)
    assert mod.inverse_conv.weight.shape == (16, 16, 33) and mod.inverse_conv._pad == (16, 16)
    mod.script_cache()
    g = golden("ts_M16.npz")
    assert np.array_equal(mod.h.numpy(), g["h"])
    assert np.abs(mod.hk.numpy() - g["hk"]).max() <= 1e-8
    assert np.abs(mod.inverse_conv.weight.detach().numpy() - g["inv_weight"]).max() <= 1e-8
    with pytest.raises(AssertionError):
        pq.PQMF(100, 12)
    pq.PQMF(100, 12, polyphase=False)
    ident = pq.PQMF(100, 16)
    ident.n_band = 1
    x = torch.zeros(1, 1, 8)
    assert ident(x) is x and ident.inverse(x) is x  # n_band == 1 is the identity (reference pqmf.py:250, :280)


@pytest.mark.parametrize("m", (2, 4, 8, 16, 32, 64))
def test_design_matches_reference_banks(pq, golden, m):
    g = golden(f"bank_M{m}.npz")
    mod = pq.PQMF(100, m)
    assert np.array_equal(mod.h.numpy(), g["h"])
    assert np.abs(mod.hk.numpy() - g["hk"]).max() <= 1e-8


def test_public_helper_names(pq):
    for name in ("reverse_half", "get_prototype", "get_qmf_bank", "kaiser_filter", "loss_wc", "center_pad_next_pow_2", "make_odd",
                 "polyphase_forward", "polyphase_inverse", "classic_forward", "classic_inverse", "PQMF", "CachedPQMF"):
        assert hasattr(pq, name)
    x = torch.arange(24.0).reshape(1, 4, 6)
    r = pq.reverse_half(x)
    assert torch.equal(r[0, 1, ::2], -x[0, 1, ::2]) and torch.equal(r[0, 1, 1::2], x[0, 1, 1::2]) and torch.equal(r[0, 0], x[0, 0])
    assert pq.center_pad_next_pow_2(torch.ones(2, 377)).shape == (2, 512)
    assert pq.make_odd(torch.ones(2, 512)).shape == (2, 513) and pq.make_odd(torch.ones(3)).shape == (3,)


def test_state_dict_roundtrip_refreshes_tables(pq):
    a = pq.CachedPQMF(100, 16)
    b = pq.CachedPQMF(80, 16)
    assert not torch.equal(a.h[:10], b.h[:10]) or a.h.shape != b.h.shape
    sd = pq.CachedPQMF(100, 16).state_dict()
    c = pq.CachedPQMF(100, 16)
    c.load_state_dict(sd)
    assert torch.equal(c.hk, a.hk)
    assert c._tables.shape == a._tables.shape


def test_torchscript_script_save_load(pq, tmp_path):
    class Wrapper(torch.nn.Module):  # same shape as the reference's PQMFWrapper (PQMFWrapper.py:17-92)
        def __init__(self):
            super().__init__()
            self.n_band = 16
            self.pqmf = pq.CachedPQMF(100, 16)

        @torch.jit.export
        def forward(self, x: torch.Tensor) -> torch.Tensor:
            if x.dim() == 2:
                x = x.unsqueeze(0)
            return self.pqmf.forward(x)

        @torch.jit.export
        def inverse(self, x: torch.Tensor) -> torch.Tensor:
            return self.pqmf.inverse(x)

    scripted = torch.jit.script(Wrapper().eval())
    path = str(tmp_path / "w.ts")
    scripted.save(path)
    loaded = torch.jit.load(path)
    assert loaded.pqmf.hk.shape == (16, 512)
    assert "pqmf_b200::analysis" in str(loaded.pqmf.forward.graph)
    scripted_plain = torch.jit.script(pq.PQMF(100, 8))  # the reference's plain PQMF is not scriptable; ours is
    assert "pqmf_b200::synthesis" in str(scripted_plain.inverse.graph)


REFERENCE = os.environ.get("PQMF_REFERENCE", "")  # a checkout of the original project (not part of this repository)


@pytest.mark.skipif(not os.path.isfile(os.path.join(REFERENCE, "PQMFWrapper.py")),
                    reason="set PQMF_REFERENCE to a checkout of the original project to run its PQMFWrapper.py")
def test_reference_wrapper_scripts_unchanged_against_dropin(tmp_path):
    """The reference's own PQMFWrapper.py, byte for byte, with dropin/ on sys.path instead of the reference's pqmf.py.
    (Copied to a temp dir at test time only because the reference checkout may be read-only and the file mkdirs next to itself.)"""
    import shutil

    shutil.copy(os.path.join(REFERENCE, "PQMFWrapper.py"), tmp_path / "PQMFWrapper.py")
    code = (
        "import sys; sys.path[:0] = [%r, %r, %r]\n"
        "import torch, PQMFWrapper as W\n"
        "import pqmf; assert 'pqmf_b200' in pqmf.CachedPQMF.__module__\n"
        "w = W.PQMFWrapper(100, 16, 8192).eval()\n"
        "s = torch.jit.script(w); s.save(%r)\n"
        "l = torch.jit.load(%r)\n"
        "assert l.get_methods() == ['forward', 'inverse', 'process']\n"
        "print('OK', l.pqmf.hk.shape)\n"
    ) % (str(tmp_path), os.path.join(ROOT, "dropin"), ROOT, str(tmp_path / "pqmf.ts"), str(tmp_path / "pqmf.ts"))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=str(tmp_path))
    assert r.returncode == 0 and "OK" in r.stdout, r.stderr[-2000:]


def test_dropin_import_names():
    code = ("import sys; sys.path[:0] = [%r, %r]\n"
            "from pqmf import CachedPQMF as A\n"
            "from PQMF.pqmf import CachedPQMF as B, PQMF, reverse_half\n"
            "assert A is B; print('OK')\n") % (os.path.join(ROOT, "dropin"), ROOT)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert r.returncode == 0 and "OK" in r.stdout, r.stderr[-2000:]


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "pseudo-quadrature-mirror-filter_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("no oracle", ""), f"{f} mentions the oracle"


def test_tables_exist_for_the_tensor_core_band_counts_and_degrade_gracefully():
    """n_band 8 / 16 / 32 get tensor-core tables (with the tap span and trim facts in the flags); banks the kernels cannot hold
    (n_band 64 at attenuation 120) and other band counts fall back to the direct form instead of raising."""
    import pqmf_b200 as pq

    assert (pq.PQMF(100, 64)._flags >> 23) & 1 and (pq.PQMF(120, 32)._flags >> 23) & 1  # split into two tap ranges
    for m, jlo, kt in ((4, 0, 128), (8, 32, 192), (16, 64, 384), (32, 128, 768)):
        mod = pq.PQMF(100, m)
        assert mod._tables.numel() > 0
        assert 32 * ((mod._flags >> 8) & 15) == jlo and 32 * ((mod._flags >> 12) & 31) == kt
        trim_a = ((mod._flags >> 17) & 7) | (((mod._flags >> 24) & 3) << 3)   # PQMF_FLAG_H4_TRIM_A
        assert 0 < trim_a <= 31 and 0 < ((mod._flags >> 20) & 7) <= 7
    for att, m in ((120, 64), (100, 2)):
        mod = pq.PQMF(att, m)
        assert mod._tables.numel() == 0 and (mod._flags >> 8) == 0


def test_cabi_argument_checks_happen_before_any_cuda_call(pq):
    """Every entry point validates its arguments on the host and returns PQMF_ERR_ARG without touching the device -- so this runs on
    the CPU box too (no compute calls without a GPU)."""
    from pqmf_b200 import _lib

    c = _lib.cabi
    c.pqmf_reconstruct_scratch_bytes.restype = ctypes.c_size_t
    c.pqmf_reconstruct_scratch_bytes.argtypes = [ctypes.c_int, ctypes.c_long, ctypes.c_long, ctypes.c_int]
    assert c.pqmf_reconstruct_scratch_bytes(0, 1024, 64, 16) == 0
    # 64 rows x 2^20: 96 MB chunks = 24 rows of 16 x 65536 floats
    assert c.pqmf_reconstruct_scratch_bytes(64, 1 << 20, 1 << 16, 16) == 24 * (1 << 20) * 4
    assert c.pqmf_reconstruct_scratch_bytes(2, 4096, 256, 16) == 2 * 4096 * 4          # a small batch is one chunk
    c.pqmf_reconstruct_f32.restype = ctypes.c_int
    c.pqmf_reconstruct_f32.argtypes = [ctypes.c_void_p] * 3 + [ctypes.c_size_t] + [ctypes.c_void_p] * 2 + [ctypes.c_int, ctypes.c_long, ctypes.c_long,
                                                                                                    ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_uint,
                                                                                                    ctypes.c_void_p]
    assert c.pqmf_reconstruct_f32(None, None, None, 0, None, None, 1, 64, 4, 16, 512, 0, 0, None) == -1
    assert c.pqmf_reconstruct_f32(None, None, None, 0, None, None, 0, 64, 4, 16, 512, 0, 0, None) == 0       # empty batch
    assert c.pqmf_analysis_pcm16(None, None, None, None, 1, 64, 2, 0, 4, 16, 512, 0, None) == -1
    assert c.pqmf_analysis_pcm16(None, None, None, None, 1, 64, 0, 0, 4, 16, 512, 0, None) == -1             # zero channels
    assert c.pqmf_synthesis_pcm16(None, None, None, None, 1, 1, 4, 16, 512, 3, 0, None) == -1                # bad delay
    assert c.pqmf_synthesis_bands_f32(None, None, None, None, 1, 4, 16, 512, 1, None, None, None, None, 0, 0, None) == -1
    assert c.pqmf_stream_step_f32(None, None, None, None, None, None, None, None, None, 1, 2048, 16, 512, 0, 0, 0, None) == -1
    assert c.pqmf_stream_step_f32(None, None, None, None, None, None, None, None, None, 1, 2049, 16, 512, 0, 0, 0, None) == -1  # T % M != 0
    devs = (ctypes.c_int * 2)(0, 1)
    assert c.pqmf_roundtrip_host_multi_f32(None, None, None, None, None, 4, 64, 16, 512, 0, 0, devs, 0) == -1     # no devices
    assert c.pqmf_roundtrip_host_multi_f32(None, None, None, None, None, 4, 64, 16, 512, 0, 0, devs, 2) == -1     # null buffers
    assert c.pqmf_roundtrip_host_pcm16(None, None, None, None, None, 4, 64, 0, 16, 512, 0, 0, 0) == -1            # zero channels
    assert b"invalid argument" in c.pqmf_strerror(-1)


def test_host_chunk_schedule_never_undercuts_the_tensor_core_kernels():
    """pqmf_host_chunk_plan (the schedule of pqmf_roundtrip_host_*): whole clips, every clip exactly once, no chunk -- ramp chunks and the
    remainder included -- below the 96 tiles of 8192 samples the Hankel kernels take (unless the whole call is smaller), none above
    the staging buffer, small chunks at the start."""
    import ctypes

    from pqmf_b200 import _lib

    f = _lib.cabi.pqmf_host_chunk_plan
    f.restype = ctypes.c_int
    f.argtypes = [ctypes.c_int, ctypes.c_long, ctypes.c_int, ctypes.POINTER(ctypes.c_long), ctypes.c_int]
    assert f(0, 4096, 1, None, 0) == -1 and f(4, 0, 1, None, 0) == -1 and f(4, 4096, 0, None, 0) == -1
    shapes = [(64, 1 << 20, 1), (64, 1 << 20, 2), (40, 1 << 16, 2), (2048, 480000, 1), (7, 65536, 2), (100, 8192, 1), (1000, 4096, 1),
              (33, 40000, 3), (5, 1 << 22, 1), (97, 70000, 1), (1, 16, 1), (3, 303104, 1), (8192, 2048, 1), (513, 131072, 2)]
    for b, t, c in shapes:
        n = f(b, t, c, None, 0)
        assert n >= 1
        buf = (ctypes.c_long * n)()
        assert f(b, t, c, buf, n) == n
        clips = list(buf)
        assert sum(clips) == b and min(clips) >= 1
        tiles_per_clip = c * -(-t // 8192)
        need = -(-96 // tiles_per_clip)
        if b >= need:
            assert min(clips) >= need, (b, t, c, clips)
        else:
            assert clips == [b]
        full = max((8 << 20) // (t * c * 4), need)
        assert max(clips) <= min(full + need - 1, b), (b, t, c, clips, full)  # a full chunk may absorb an undersized remainder
        if n >= 8:  # long schedules start and end with small chunks (pipeline fill and drain)
            assert clips[0] < max(clips) or full == need


def test_host_chunk_schedule_with_tiny_chunks():
    """The same properties when PQMF_HOST_CHUNK_MIB makes a chunk no larger than the kernels' minimum (the setting is read once per
    process: a subprocess), on random shapes: a remainder below the minimum joins the chunk before it instead of running alone."""
    import subprocess
    import textwrap

    code = textwrap.dedent("""
        import ctypes, random, sys
        sys.path.insert(0, %r)
        from pqmf_b200 import _lib
        f = _lib.cabi.pqmf_host_chunk_plan
        f.restype = ctypes.c_int
        f.argtypes = [ctypes.c_int, ctypes.c_long, ctypes.c_int, ctypes.POINTER(ctypes.c_long), ctypes.c_int]
        random.seed(7)
        for _ in range(1500):
            b = random.randint(1, 3000); t = random.choice((2048, 4096, 8192, 40960, 65536, 303104, 1 << 20)); c = random.choice((1, 2, 3))
            n = f(b, t, c, None, 0)
            buf = (ctypes.c_long * n)()
            assert f(b, t, c, buf, n) == n
            clips = list(buf)
            need = -(-96 // (c * -(-t // 8192)))
            full = max((1 << 20) // (t * c * 4), need)
            assert sum(clips) == b
            assert min(clips) >= need or clips == [b], (b, t, c, clips[-4:], need)
            assert max(clips) <= min(full + need - 1, b), (b, t, c, max(clips), full, need)
        print("ok")
    """) % ROOT
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, PQMF_HOST_CHUNK_MIB="1"), capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stderr[-2000:]
