"""Loads the in-tree native libraries and fails loudly when they are missing.

* ``libpqmf_b200.so``       -- sm_100a kernels behind the C ABI of include/pqmf_b200.h (ctypes handle: ``cabi``)
* ``libpqmf_b200_torch.so`` -- ``torch.ops.pqmf_b200.*`` (CUDA dispatch key only: CPU tensors raise)

There is no CPU fallback and no alternative backend: if either library cannot be loaded the import of
``pqmf_b200`` raises, pointing at the build command.
"""
from __future__ import annotations

import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
_CABI_PATH = os.path.join(_HERE, "libpqmf_b200.so")
_TORCH_PATH = os.path.join(_HERE, "libpqmf_b200_torch.so")
_BUILD_HINT = "build it with:  python -c 'import __graft_entry__ as g; g.build()'   (or make -C {}/csrc all torch)".format(_HERE)

PQMF_ERR_UNSUPPORTED = -2
PQMF_FLAG_EXACT = 1
PQMF_FLAG_NO_SIGN = 2
PQMF_FLAG_FOLD = 4
PQMF_FLAG_NO_PAIR = 8
PQMF_FLAG_FP32 = 16
PQMF_FLAG_NO_FOLD = 32
PQMF_FLAG_H4_SPLIT = 1 << 23
PQMF_DTYPE_F32 = 0
PQMF_DTYPE_F16 = 1
PQMF_DTYPE_BF16 = 2


def _load():
    for path in (_CABI_PATH, _TORCH_PATH):
        if not os.path.exists(path):
            raise ImportError(f"pqmf_b200: native library missing: {path}\n{_BUILD_HINT}")
    try:
        lib = ctypes.CDLL(_CABI_PATH, mode=ctypes.RTLD_GLOBAL)
    except OSError as e:  # pragma: no cover
        raise ImportError(f"pqmf_b200: cannot load {_CABI_PATH}: {e}\n{_BUILD_HINT}") from e
    try:
        torch.ops.load_library(_TORCH_PATH)
    except Exception as e:  # pragma: no cover
        raise ImportError(f"pqmf_b200: cannot load {_TORCH_PATH}: {e}\n{_BUILD_HINT}") from e
    return lib


cabi = _load()

_f32p = ctypes.POINTER(ctypes.c_float)
_vp = ctypes.c_void_p

cabi.pqmf_abi_version.restype = ctypes.c_int
cabi.pqmf_strerror.restype = ctypes.c_char_p
cabi.pqmf_strerror.argtypes = [ctypes.c_int]
cabi.pqmf_launch_count.restype = ctypes.c_ulonglong
cabi.pqmf_path_for.restype = ctypes.c_int
cabi.pqmf_path_for.argtypes = [ctypes.c_int, ctypes.c_int, _vp, ctypes.c_uint]
cabi.pqmf_tables_numel.restype = ctypes.c_long
cabi.pqmf_tables_numel.argtypes = [ctypes.c_int, ctypes.c_int]
cabi.pqmf_build_tables_f32.restype = ctypes.c_int
cabi.pqmf_build_tables_f32.argtypes = [_vp, _vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp, ctypes.POINTER(ctypes.c_double),
                                       ctypes.POINTER(ctypes.c_uint)]
cabi.pqmf_analysis_f32.restype = ctypes.c_int
cabi.pqmf_analysis_f32.argtypes = [_vp, _vp, _vp, _vp, ctypes.c_int, ctypes.c_long, ctypes.c_long, ctypes.c_int, ctypes.c_int,
                                   ctypes.c_uint, _vp]
cabi.pqmf_synthesis_f32.restype = ctypes.c_int
cabi.pqmf_synthesis_f32.argtypes = [_vp, _vp, _vp, _vp, ctypes.c_int, ctypes.c_long, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                    ctypes.c_uint, _vp]
cabi.pqmf_analysis_stream_f32.restype = ctypes.c_int
cabi.pqmf_analysis_stream_f32.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, ctypes.c_int, ctypes.c_long, ctypes.c_int, ctypes.c_int,
                                          ctypes.c_int, ctypes.c_uint, _vp]
cabi.pqmf_synthesis_stream_f32.restype = ctypes.c_int
cabi.pqmf_synthesis_stream_f32.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, ctypes.c_int, ctypes.c_long, ctypes.c_int, ctypes.c_int,
                                           ctypes.c_int, ctypes.c_uint, _vp]
cabi.pqmf_analysis_pcm16.restype = ctypes.c_int
cabi.pqmf_analysis_pcm16.argtypes = [_vp, _vp, _vp, _vp, ctypes.c_int, ctypes.c_long, ctypes.c_int, ctypes.c_int, ctypes.c_long, ctypes.c_int,
                                     ctypes.c_int, ctypes.c_uint, _vp]
cabi.pqmf_synthesis_pcm16.restype = ctypes.c_int
cabi.pqmf_synthesis_pcm16.argtypes = [_vp, _vp, _vp, _vp, ctypes.c_int, ctypes.c_int, ctypes.c_long, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                      ctypes.c_uint, _vp]
cabi.pqmf_roundtrip_host_f32.restype = ctypes.c_int
cabi.pqmf_roundtrip_host_f32.argtypes = [_vp, _vp, _vp, _vp, _vp, ctypes.c_int, ctypes.c_long, ctypes.c_int, ctypes.c_int,
                                         ctypes.c_int, ctypes.c_uint, ctypes.c_int]
cabi.pqmf_stream_step_f32.restype = ctypes.c_int
cabi.pqmf_stream_step_f32.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, ctypes.c_int, ctypes.c_long, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                      ctypes.c_int, ctypes.c_uint, _vp]
cabi.pqmf_synthesis_bands_f32.restype = ctypes.c_int
cabi.pqmf_synthesis_bands_f32.argtypes = [_vp, _vp, _vp, _vp, ctypes.c_int, ctypes.c_long, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp, _vp, _vp, _vp,
                                          ctypes.c_int, ctypes.c_uint, _vp]
cabi.pqmf_roundtrip_host_pcm16.restype = ctypes.c_int
cabi.pqmf_roundtrip_host_pcm16.argtypes = [_vp, _vp, _vp, _vp, _vp, ctypes.c_int, ctypes.c_long, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                           ctypes.c_int, ctypes.c_uint, ctypes.c_int]
cabi.pqmf_roundtrip_host_multi_f32.restype = ctypes.c_int
cabi.pqmf_roundtrip_host_multi_f32.argtypes = [_vp, _vp, _vp, _vp, _vp, ctypes.c_int, ctypes.c_long, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                               ctypes.c_uint, ctypes.POINTER(ctypes.c_int), ctypes.c_int]
# half-precision I/O (dtype: PQMF_DTYPE_*); PQMF_ERR_UNSUPPORTED where no native kernel exists
cabi.pqmf_analysis_x.restype = ctypes.c_int
cabi.pqmf_analysis_x.argtypes = [_vp, _vp, _vp, _vp, ctypes.c_int, ctypes.c_long, ctypes.c_long, ctypes.c_int, ctypes.c_int, ctypes.c_uint,
                                 ctypes.c_int, _vp]
cabi.pqmf_synthesis_x.restype = ctypes.c_int
cabi.pqmf_synthesis_x.argtypes = [_vp, _vp, _vp, _vp, ctypes.c_int, ctypes.c_long, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_uint,
                                  ctypes.c_int, _vp]
cabi.pqmf_roundtrip_x.restype = ctypes.c_int
cabi.pqmf_roundtrip_x.argtypes = [_vp, _vp, _vp, _vp, _vp, ctypes.c_int, ctypes.c_long, ctypes.c_long, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                  ctypes.c_uint, ctypes.c_int, _vp]
cabi.pqmf_reconstruct_scratch_bytes.restype = ctypes.c_size_t
cabi.pqmf_reconstruct_scratch_bytes.argtypes = [ctypes.c_int, ctypes.c_long, ctypes.c_long, ctypes.c_int]
cabi.pqmf_reconstruct_x.restype = ctypes.c_int
cabi.pqmf_reconstruct_x.argtypes = [_vp, _vp, _vp, ctypes.c_size_t, _vp, _vp, ctypes.c_int, ctypes.c_long, ctypes.c_long, ctypes.c_int, ctypes.c_int,
                                    ctypes.c_int, ctypes.c_uint, ctypes.c_int, _vp]

if cabi.pqmf_abi_version() != 2:  # pragma: no cover
    raise ImportError("pqmf_b200: libpqmf_b200.so ABI version mismatch; rebuild")


def strerror(code: int) -> str:
    return cabi.pqmf_strerror(int(code)).decode()


def check(code: int, what: str) -> None:
    if code != 0:
        raise RuntimeError(f"{what} failed: {strerror(code)} (code {code})")


def launch_count() -> int:
    """Kernels launched by libpqmf_b200.so in this process."""
    return int(cabi.pqmf_launch_count())


def library_paths():
    return [_CABI_PATH, _TORCH_PATH]


def build_tables(hk: torch.Tensor, h: torch.Tensor):
    """Host-side factorisation hk ~= g (x) C for the fast path.  Returns (tables fp32 CPU tensor, residual,
    fast_flags); an empty tensor when (n_band, L) has no fast path."""
    m, length = int(hk.shape[0]), int(hk.shape[1])
    n = cabi.pqmf_tables_numel(m, length)
    if n <= 0:
        return torch.zeros(0, dtype=torch.float32), float("nan"), 0
    hk_c = hk.detach().to("cpu", torch.float32).contiguous()
    h_c = h.detach().to("cpu", torch.float32).contiguous()
    out = torch.empty(n, dtype=torch.float32)
    res = ctypes.c_double(0.0)
    fast_flags = ctypes.c_uint(0)
    rc = cabi.pqmf_build_tables_f32(hk_c.data_ptr(), h_c.data_ptr(), int(h_c.numel()), m, length, out.data_ptr(),
                                    ctypes.byref(res), ctypes.byref(fast_flags))
    if rc == PQMF_ERR_UNSUPPORTED:  # e.g. a bank too long for one SM's shared memory (n_band 32 at attenuation 120): direct form
        return torch.zeros(0, dtype=torch.float32), float("nan"), 0
    check(rc, "pqmf_build_tables_f32")
    return out, float(res.value), int(fast_flags.value)
