"""float16 / bfloat16 signals and sub-bands: every call returns its input's dtype and is bit-equal to the float32 call on the widened
input followed by a round-to-nearest-even cast -- on the native half-precision Hankel-4 kernels (large offline calls) and on the
staged path (widen, fp32 kernels, round) alike.  Also module casts, autograd, TorchScript and the dtype errors."""
import pytest
import torch

pytestmark = pytest.mark.gpu

HALF = [torch.bfloat16, torch.float16]
NATIVE = (16, 1, 1 << 16)  # 16 rows x 8 tiles of 8192 samples: >= 96 tiles


@pytest.fixture(scope="module")
def pq():
    import pqmf_b200

    return pqmf_b200


def signal(shape, dtype, seed=0, scale=0.5):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (scale * torch.randn(shape, generator=g, device="cuda")).clamp_(-1, 1).to(dtype)


def same_bits(a, b):
    assert a.dtype == b.dtype and a.shape == b.shape, (a.dtype, b.dtype, a.shape, b.shape)
    return torch.equal(a.view(torch.int16), b.view(torch.int16))


def dtype_code(dtype):
    from pqmf_b200 import _lib

    return {torch.float16: _lib.PQMF_DTYPE_F16, torch.bfloat16: _lib.PQMF_DTYPE_BF16}[dtype]


def rc_analysis(mod, x, n_frames):
    """return code of pqmf_analysis_x for this module and input: 0 = the native half-precision kernels ran"""
    from pqmf_b200 import _lib

    hk = mod.hk.float().contiguous()
    m, length = hk.shape
    y = torch.empty(x.shape[0], x.shape[1] * m, n_frames, dtype=x.dtype, device=x.device)
    rc = _lib.cabi.pqmf_analysis_x(x.data_ptr(), y.data_ptr(), hk.data_ptr(), mod._tables.data_ptr() if mod._tables.numel() else None,
                                   x.shape[0] * x.shape[1], x.shape[-1], n_frames, m, length, mod._flags, dtype_code(x.dtype),
                                   torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return rc


def rc_synthesis(mod, s, delay):
    from pqmf_b200 import _lib

    hk = mod.hk.float().contiguous()
    m, length = hk.shape
    out = torch.empty(s.shape[0], s.shape[1] // m, m * s.shape[-1], dtype=s.dtype, device=s.device)
    rc = _lib.cabi.pqmf_synthesis_x(s.data_ptr(), out.data_ptr(), hk.data_ptr(), mod._tables.data_ptr() if mod._tables.numel() else None,
                                    s.shape[0] * (s.shape[1] // m), s.shape[-1], m, length, delay, mod._flags, dtype_code(s.dtype),
                                    torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return rc


def check_both_directions(mod, x):
    y = mod(x)
    assert y.dtype == x.dtype
    assert same_bits(y, mod(x.float()).to(x.dtype))
    out = mod.inverse(y)
    assert out.dtype == x.dtype
    assert same_bits(out, mod.inverse(y.float()).to(x.dtype))
    return y


# ---------------------------------------------------------------- 1. native path
@pytest.mark.parametrize("dtype", HALF)
@pytest.mark.parametrize("n_band", [4, 8, 16, 32])
@pytest.mark.parametrize("cls", ["PQMF", "CachedPQMF"])
@pytest.mark.parametrize("exact", [False, True])
def test_native_path_bit_identical(pq, dtype, n_band, cls, exact):
    mod = getattr(pq, cls)(100, n_band, exact=exact).cuda()
    x = signal(NATIVE, dtype, seed=n_band)
    y = check_both_directions(mod, x)
    # the half-precision kernels really ran (a silent fallback would pass the bit-identity check as well)
    assert rc_analysis(mod, x, NATIVE[-1] // n_band) == 0
    assert rc_synthesis(mod, y, 1 if cls == "CachedPQMF" else 0) == 0


# ---------------------------------------------------------------- 2. staged path
@pytest.mark.parametrize("dtype", HALF)
@pytest.mark.parametrize("case", ["small_batch", "ragged", "t_not_8", "f_not_4", "n_band_2", "n_band_64_split", "exact_small", "fp32",
                                  "check_range"])
def test_staged_path_bit_identical(pq, dtype, case):
    kwargs, cls, n_band, shape = {}, "PQMF", 16, NATIVE
    if case == "small_batch":        # n_band 16 fold kernels
        shape = (2, 1, 16384)
    elif case == "ragged":           # CachedPQMF: T % n_band != 0 -> ceil(T / n_band) frames
        cls, shape = "CachedPQMF", (16, 1, (1 << 16) - 5)
    elif case == "t_not_8":
        cls, n_band, shape = "CachedPQMF", 4, (16, 1, (1 << 16) - 4)
    elif case == "f_not_4":          # analysis native (T % 8 == 0), synthesis staged (F % 4 == 2)
        shape = (16, 1, (1 << 16) - 32)
    elif case == "n_band_2":         # no tables: direct form
        n_band, shape = 2, (4, 1, 8192)
    elif case == "n_band_64_split":  # bank in two tap ranges
        n_band = 64
    elif case == "exact_small":
        kwargs, shape = {"exact": True}, (2, 1, 16384)
    elif case == "fp32":
        kwargs, shape = {"fp32": True}, (2, 1, 16384)
    else:
        kwargs = {"check_range": True}
    mod = getattr(pq, cls)(100, n_band, **kwargs).cuda()
    x = signal(shape, dtype, seed=3)
    y = check_both_directions(mod, x)
    if case == "n_band_64_split":
        assert mod._flags & pq._lib.PQMF_FLAG_H4_SPLIT
        assert rc_analysis(mod, x, NATIVE[-1] // 64) == pq._lib.PQMF_ERR_UNSUPPORTED
    if case == "f_not_4":
        assert rc_analysis(mod, x, x.shape[-1] // 16) == 0
        assert rc_synthesis(mod, y, 0) == pq._lib.PQMF_ERR_UNSUPPORTED


@pytest.mark.parametrize("dtype", HALF)
def test_check_range_routes_out_of_range_half_input_to_fp32(pq, dtype):
    mod = pq.PQMF(100, 16, check_range=True).cuda()
    x = signal(NATIVE, dtype, seed=4) * 1e-7  # below the range the tensor-core kernels are meant for
    assert same_bits(mod(x), mod(x.float()).to(dtype))


@pytest.mark.parametrize("dtype", HALF)
def test_misaligned_base_pointer(pq, dtype):
    mod = pq.PQMF(100, 16).cuda()
    n = NATIVE[0] * NATIVE[-1]
    flat = signal((n + 8,), dtype, seed=5)
    x = flat[1:1 + n].view(NATIVE)  # contiguous, 2 bytes past a 16-byte boundary
    assert x.is_contiguous() and x.data_ptr() % 16 != 0
    assert rc_analysis(mod, x, NATIVE[-1] // 16) == pq._lib.PQMF_ERR_UNSUPPORTED
    check_both_directions(mod, x)
    flat_s = mod(signal(NATIVE, dtype, seed=6)).flatten()
    s = torch.empty(flat_s.numel() + 8, dtype=dtype, device="cuda")
    s[1:1 + flat_s.numel()] = flat_s
    s = s[1:1 + flat_s.numel()].view(NATIVE[0], 16, -1)
    assert rc_synthesis(mod, s, 0) == pq._lib.PQMF_ERR_UNSUPPORTED
    assert same_bits(mod.inverse(s), mod.inverse(s.float()).to(dtype))


@pytest.mark.parametrize("dtype", HALF)
def test_free_functions(pq, dtype):
    mod = pq.PQMF(100, 8).cuda()
    hk = mod.hk
    for shape in [(2, 1, 8192), NATIVE]:
        x = signal(shape, dtype, seed=7)
        for fn in (pq.polyphase_forward, pq.classic_forward):
            y = fn(x, hk)
            assert same_bits(y, fn(x.float(), hk).to(dtype))
        for fn in (pq.polyphase_inverse, pq.classic_inverse):
            out = fn(y, hk)
            assert same_bits(out, fn(y.float(), hk).to(dtype))
    # a half-precision bank is used as it is (rounded), in fp32
    hb = hk.to(dtype)
    assert same_bits(pq.classic_forward(x, hb), pq.classic_forward(x.float(), hb.float()).to(dtype))


# ---------------------------------------------------------------- 3. process / reconstruct
@pytest.mark.parametrize("dtype", HALF)
@pytest.mark.parametrize("cls", ["PQMF", "CachedPQMF"])
@pytest.mark.parametrize("shape", [NATIVE, (2, 1, 16384), (400, 1, 1 << 16), (390, 1, 1 << 16)])
def test_process_and_reconstruct(pq, dtype, cls, shape):
    mod = getattr(pq, cls)(100, 16).cuda()
    x = signal(shape, dtype, seed=8)
    out, y = mod.process(x)
    y_ref = mod(x)
    assert same_bits(y, y_ref)
    assert same_bits(out, mod.inverse(y_ref))  # the synthesis reads the rounded sub-bands
    assert same_bits(mod.reconstruct(x), out)


# ---------------------------------------------------------------- 4. module casts
@pytest.mark.parametrize("dtype", HALF)
@pytest.mark.parametrize("n_band", [8, 16])
def test_half_module_uses_the_rounded_bank(pq, dtype, n_band):
    half = pq.CachedPQMF(100, n_band).cuda().to(dtype)
    assert half.hk.dtype == dtype and half.h.dtype == dtype and half._tables.dtype == torch.float32
    ref = pq.CachedPQMF(100, n_band).cuda()
    with torch.no_grad():
        ref.hk.copy_(half.hk.float())
        ref.h.copy_(half.h.float())
    ref.refresh_tables()
    assert torch.equal(half._tables.view(torch.int32), ref._tables.view(torch.int32)) and half._flags == ref._flags
    for shape in [NATIVE, (2, 1, 16384)]:
        for in_dtype in (torch.float32, dtype):  # input dtype and module dtype are independent
            x = signal(shape, in_dtype, seed=9)
            y = half(x)
            assert y.dtype == in_dtype and same_bits(y, ref(x))
            assert same_bits(half.inverse(y), ref.inverse(y))


def test_half_float_cast_and_device_move(pq):
    mod = pq.PQMF(100, 16)
    tables = mod._tables.clone()
    mod = mod.cuda()
    assert torch.equal(mod._tables.cpu().view(torch.int32), tables.view(torch.int32))  # a device move keeps the tables
    back = pq.PQMF(100, 16).cuda().half().float()
    fresh = pq.PQMF(100, 16).cuda()
    with torch.no_grad():
        fresh.hk.copy_(back.hk)
        fresh.h.copy_(back.h)
    fresh.refresh_tables()
    x = signal(NATIVE, torch.float32, seed=10)
    assert torch.equal(back(x), fresh(x)) and torch.equal(back.inverse(back(x)), fresh.inverse(fresh(x)))


# ---------------------------------------------------------------- 5. autograd
def _ulp(v, dtype):
    """spacing of `dtype` at |v| (v float32)"""
    mant, tiny = (10, 2.0 ** -14) if dtype == torch.float16 else (7, 2.0 ** -126)
    e = torch.floor(torch.log2(v.abs().clamp_min(tiny)))
    return torch.exp2(e - mant)


@pytest.mark.parametrize("dtype", HALF)
@pytest.mark.parametrize("direction", ["analysis", "synthesis"])
@pytest.mark.parametrize("mag", [1e-4, 1e-2, 1.0, 1e3])
def test_autograd(pq, dtype, direction, mag):
    mod = pq.PQMF(100, 16).cuda()
    if direction == "analysis":
        inp = signal(NATIVE, dtype, seed=11)
        fn = mod.forward
        g_shape = (NATIVE[0], 16, NATIVE[-1] // 16)
    else:
        inp = mod(signal(NATIVE, dtype, seed=12))
        fn = mod.inverse
        g_shape = NATIVE
    gen = torch.Generator(device="cuda").manual_seed(13)
    g = (mag * (2 * torch.rand(g_shape, generator=gen, device="cuda") - 1)).to(dtype)
    x = inp.clone().requires_grad_(True)
    fn(x).backward(g)
    x32 = inp.float().requires_grad_(True)
    fn(x32).backward(g.float())
    assert x.grad.dtype == dtype
    a, b = x.grad.float(), x32.grad
    finite = b.abs() < torch.finfo(dtype).max
    assert finite.float().mean() > 0.99
    err = (a - b).abs()[finite]
    tol = torch.maximum(_ulp(a, dtype), _ulp(b, dtype))[finite]
    assert bool((err <= tol).all()), float((err / tol).max())


# ---------------------------------------------------------------- 6. TorchScript
def test_torchscript_cached_pqmf_bf16(pq):
    mod = pq.CachedPQMF(100, 16).cuda()
    scripted = torch.jit.script(mod)
    for shape in [NATIVE, (2, 1, 16384)]:
        x = signal(shape, torch.bfloat16, seed=14)
        y = scripted(x)
        assert same_bits(y, mod(x)) and same_bits(scripted.inverse(y), mod.inverse(y))
    half = torch.jit.script(pq.PQMF(100, 16).cuda().half())
    x = signal(NATIVE, torch.float16, seed=15)
    assert half(x).dtype == torch.float16


# ---------------------------------------------------------------- 7. errors
def test_unsupported_dtypes_and_entry_points_raise(pq):
    mod = pq.CachedPQMF(100, 16).cuda()
    with pytest.raises(RuntimeError, match="Double"):
        mod(torch.zeros(2, 1, 4096, dtype=torch.float64, device="cuda"))
    with pytest.raises(RuntimeError, match="Double"):
        mod.inverse(torch.zeros(2, 16, 256, dtype=torch.float64, device="cuda"))
    x = signal((4, 1, 4096), torch.bfloat16)
    s = signal((4, 16, 256), torch.float16)
    with pytest.raises(RuntimeError, match="BFloat16"):
        mod.forward_stream(x)
    with pytest.raises(RuntimeError, match="Half"):
        mod.inverse_stream(s)
    with pytest.raises(RuntimeError, match="BFloat16"):
        mod.process_stream(x)
    with pytest.raises(RuntimeError, match="Half"):
        mod.inverse_pcm16(s)
    with pytest.raises(RuntimeError, match="Half"):
        mod.inverse_bands([s[:, k] for k in range(16)], 256, torch.zeros(0, device="cuda"), torch.zeros(0, device="cuda"),
                          torch.zeros(0, device="cuda"))
