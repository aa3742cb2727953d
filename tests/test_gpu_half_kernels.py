"""The native float16 / bfloat16 Hankel-4 kernels where they can go wrong: the steady state of the persistent loop (several tiles per
CTA, so the one-tile-ahead prefetch, the double buffers and the barrier phases all wrap), odd tile counts (the CTA pair's padding
tile), partial last tiles, the scalar fallbacks of the half-precision stores, and every bank the half kernels serve (attenuation
50 to 140, n_band 4 to 64).  Every case checks that the native kernels really ran, that the result is bit-equal to the float32
call on the widened input rounded to nearest even, and -- independently of the float32 kernels -- that excerpts agree with the
float64 oracle within the float32 tolerance plus half an ulp of the output dtype."""
import pytest
import torch

from oracle import pqmf_oracle as O

pytestmark = pytest.mark.gpu

HALF = [torch.bfloat16, torch.float16]
CLASSES = ["PQMF", "CachedPQMF"]
TOL = 1e-5
TILE = 8192  # samples per tile of the Hankel-4 kernels
ATTENUATIONS = [50, 60, 80, 120, 140]
# banks the host table builder splits into two tap ranges (staged path for half precision), and banks without tables (direct form)
SPLIT = {(60, 64), (80, 64), (120, 32), (140, 32)}
NO_TABLES = {(120, 64), (140, 64)}


@pytest.fixture(scope="module")
def pq():
    import pqmf_b200

    return pqmf_b200


@pytest.fixture(scope="module")
def bank(pq):
    """modules by (class, attenuation, n_band): the prototype design runs scipy's fmin on the host"""
    cache = {}

    def get(cls, attenuation, n_band):
        key = (cls, attenuation, n_band)
        if key not in cache:
            cache[key] = getattr(pq, cls)(attenuation, n_band).cuda()
        return cache[key]

    return get


def signal(shape, dtype, seed=0, scale=0.5):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (scale * torch.randn(shape, generator=g, device="cuda")).clamp_(-1, 1).to(dtype)


def same_bits(a, b):
    assert a.dtype == b.dtype and a.shape == b.shape, (a.dtype, b.dtype, a.shape, b.shape)
    if a.dtype == torch.float32:
        return torch.equal(a.view(torch.int32), b.view(torch.int32))
    return torch.equal(a.view(torch.int16), b.view(torch.int16))


def dtype_code(dtype):
    from pqmf_b200 import _lib

    return {torch.float16: _lib.PQMF_DTYPE_F16, torch.bfloat16: _lib.PQMF_DTYPE_BF16}[dtype]


def tables_ptr(mod):
    return mod._tables.data_ptr() if mod._tables.numel() else None


def rc_analysis(mod, x, n_frames):
    """return code of pqmf_analysis_x for this module and input: 0 = the native half-precision kernels ran"""
    from pqmf_b200 import _lib

    hk = mod.hk.float().contiguous()
    m, length = hk.shape
    y = torch.empty(x.shape[0], x.shape[1] * m, n_frames, dtype=x.dtype, device=x.device)
    rc = _lib.cabi.pqmf_analysis_x(x.data_ptr(), y.data_ptr(), hk.data_ptr(), tables_ptr(mod), x.shape[0] * x.shape[1], x.shape[-1],
                                   n_frames, m, length, mod._flags, dtype_code(x.dtype), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return rc


def rc_synthesis(mod, s, delay):
    from pqmf_b200 import _lib

    hk = mod.hk.float().contiguous()
    m, length = hk.shape
    out = torch.empty(s.shape[0], s.shape[1] // m, m * s.shape[-1], dtype=s.dtype, device=s.device)
    rc = _lib.cabi.pqmf_synthesis_x(s.data_ptr(), out.data_ptr(), hk.data_ptr(), tables_ptr(mod), s.shape[0] * (s.shape[1] // m),
                                    s.shape[-1], m, length, delay, mod._flags, dtype_code(s.dtype), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return rc


def taps(flags):
    """(jlo, kt) of the bank's Hankel-4 images (PQMF_FLAG_TAPS)"""
    return 32 * ((flags >> 8) & 0xF), 32 * ((flags >> 12) & 0x1F)


def _ulp(v, dtype):
    """spacing of `dtype` at |v|"""
    mant, tiny = (10, 2.0 ** -14) if dtype == torch.float16 else (7, 2.0 ** -126)
    e = torch.floor(torch.log2(v.abs().clamp_min(tiny)))
    return torch.exp2(e - mant)


def assert_near_oracle(q, ref, tol32, dtype, what):
    """|q - ref| <= tol32 + ulp(|ref| + tol32) / 2: the float32 kernels' bound plus the final rounding to `dtype`"""
    q, ref = torch.from_numpy(q), torch.from_numpy(ref)
    bound = tol32 + (_ulp(ref.abs() + tol32, dtype) / 2 if dtype in HALF else 0.0)
    err = (q - ref).abs()
    assert bool((err <= bound).all()), f"{what}: worst |error| / bound = {float((err / bound).max()):.3g}"


def oracle_excerpt(x_row, y_row, out_row, hk, delay, start, n, dtype):
    """Frames [start, start + n) of one row's sub-bands, and the output samples of those frames, against the float64 oracle run
    on the cropped input they depend on (filtering is local): one filter length of halo on each side, cut at an even frame (the
    sign mask follows the global frame parity), or at the row's own ends.  The synthesis oracle reads the sub-bands the kernel
    produced (widened)."""
    m, length = hk.shape
    n_frames = y_row.shape[1]
    halo = length // m
    f0 = max(0, start - halo) & ~1
    f1 = min(n_frames, start + n + halo)
    tol_a, tol_s = TOL / 2, (TOL if m == 64 else TOL / 2)  # n_band 64 synthesis: fp32 accumulation alone is ~4e-6
    y64 = O.analysis(x_row[f0 * m:f1 * m][None], hk)[0]
    assert_near_oracle(y_row[:, start:start + n], y64[:, start - f0:start - f0 + n], tol_a, dtype, f"analysis, frames {start}+{n}")
    o64 = O.synthesis(y_row[:, f0:f1][None], hk, delay_frames=delay)[0]
    a = (start - f0) * m
    assert_near_oracle(out_row[start * m:(start + n) * m], o64[a:a + n * m], tol_s, dtype, f"synthesis, frames {start}+{n}")


def oracle_rows(mod, x, y, out, delay, rows):
    """Excerpts of the given rows: the row start, tile boundaries (the second tile, one in the middle, the last) and the row end."""
    hk = mod.hk.cpu().numpy()
    m = hk.shape[0]
    n_frames = y.shape[-1]
    n = 4096 // m  # frames of 4096 samples: half a tile
    fpt = TILE // m
    tiles_per_row = -(-n_frames * m // TILE)
    starts = [0, fpt - n // 2, (tiles_per_row // 2) * fpt - n // 2, (tiles_per_row - 1) * fpt - n // 2, n_frames - n]
    for r in rows:
        xr = x[r, 0].double().cpu().numpy()
        yr = y[r].double().cpu().numpy()
        orow = out[r, 0].double().cpu().numpy()
        for s in starts:
            oracle_excerpt(xr, yr, orow, hk, delay, s, n, x.dtype)


def check_call(pq, mod, x, delay, rc_a, rc_s, rows):
    """Both directions: the expected route (rc 0 = native, PQMF_ERR_UNSUPPORTED = staged), bit-identity with the float32 call on
    the widened input, and oracle excerpts of `rows`."""
    m = mod.n_band
    n_frames = x.shape[-1] // m
    assert rc_analysis(mod, x, n_frames) == rc_a
    y = mod(x)
    assert y.dtype == x.dtype and y.shape == (x.shape[0], m, n_frames)
    assert same_bits(y, mod(x.float()).to(x.dtype))
    assert rc_synthesis(mod, y, delay) == rc_s
    out = mod.inverse(y)
    assert out.dtype == x.dtype
    assert same_bits(out, mod.inverse(y.float()).to(x.dtype))
    oracle_rows(mod, x, y, out, delay, rows)


# ---------------------------------------------------------------- 1. steady state of the persistent loop
# 37 rows x (33 tiles - 12 frames): 1221 tiles, odd, ~8 per CTA on 148 SMs; the last tile of a row is partial, T % 8 == 0 and
# F % 4 == 0, so both directions run natively.  Tiles of rows >= 5 are second or later iterations of their CTA.
def steady_shape(m):
    return (37, 1, 33 * TILE - 12 * m)


@pytest.mark.parametrize("cls", CLASSES)
@pytest.mark.parametrize("dtype", HALF)
@pytest.mark.parametrize("n_band", [4, 8, 16, 32])
def test_steady_state(pq, bank, n_band, dtype, cls):
    mod = bank(cls, 100, n_band)
    x = signal(steady_shape(n_band), dtype, seed=n_band)
    check_call(pq, mod, x, 1 if cls == "CachedPQMF" else 0, 0, 0, rows=(0, 5, 18, 36))


# ---------------------------------------------------------------- 2. every bank the half-precision kernels serve
# 13 rows x (29 tiles - 8 frames): 377 tiles, odd, 2-3 per CTA.  n_band 4 runs both classes: their synthesis offsets select the two
# synthesis images (test_n_band_4_sweep_hits_both_synthesis_images); other band counts alternate the class over the sweep.
def sweep():
    cases = []
    for i, att in enumerate(ATTENUATIONS):
        for j, m in enumerate([4, 8, 16, 32, 64]):
            if (att, m) not in NO_TABLES:
                cases += [(att, m, cls) for cls in (CLASSES if m == 4 else [CLASSES[(i + j) % 2]])]
    return cases


@pytest.mark.parametrize("dtype", HALF)
@pytest.mark.parametrize("attenuation,n_band,cls", sweep())
def test_every_bank(pq, bank, attenuation, n_band, cls, dtype):
    mod = bank(cls, attenuation, n_band)
    assert mod._tables.numel() > 0
    split = (attenuation, n_band) in SPLIT
    assert bool(mod._flags & pq._lib.PQMF_FLAG_H4_SPLIT) == split
    rc = pq._lib.PQMF_ERR_UNSUPPORTED if split else 0  # split banks: two launches, the second accumulating -- staged
    x = signal((13, 1, 29 * TILE - 8 * n_band), dtype, seed=attenuation + n_band)
    check_call(pq, mod, x, 1 if cls == "CachedPQMF" else 0, rc, rc, rows=(0, 6, 12))


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


@pytest.mark.parametrize("cls", CLASSES)
def test_fp32_unsplit_n_band_64(pq, bank, cls):
    """Attenuation 50 is the one n_band-64 bank that fits one SM unsplit: the float32 Hankel-4 launch at M = 64."""
    mod = bank(cls, 50, 64)
    length = mod.hk.shape[1]
    assert length == 1024 and taps(mod._flags) == (128, 768) and not mod._flags & pq._lib.PQMF_FLAG_H4_SPLIT
    assert pq._lib.cabi.pqmf_path_for(64, length, tables_ptr(mod), mod._flags) == 1
    x = signal((13, 1, 29 * TILE - 8 * 64), torch.float32, seed=64)
    y = mod(x)
    out = mod.inverse(y)
    oracle_rows(mod, x, y, out, 1 if cls == "CachedPQMF" else 0, rows=(0, 6, 12))


# ---------------------------------------------------------------- 3. scalar fallbacks of the half-precision analysis store
# The vector stores need F % 8 == 0 (n_band 4 and 8), F % 2 == 0 (n_band 32).  41 rows x 9 tiles = 369 tiles.  Synthesis is native
# exactly where F % 4 == 0.
@pytest.mark.parametrize("dtype", HALF)
@pytest.mark.parametrize("n_band,n_frames", [(4, 18426), (4, 18428), (4, 18430), (8, 9212), (8, 9213), (32, 2303), (32, 2301)])
def test_store_fallbacks(pq, bank, n_band, n_frames, dtype):
    mod = bank("PQMF", 100, n_band)
    x = signal((41, 1, n_frames * n_band), dtype, seed=n_frames)
    rc_s = 0 if n_frames % 4 == 0 else pq._lib.PQMF_ERR_UNSUPPORTED
    check_call(pq, mod, x, 0, 0, rc_s, rows=(0, 40))


# ---------------------------------------------------------------- 4. process / reconstruct against the float32 calls
@pytest.mark.parametrize("cls", CLASSES)
@pytest.mark.parametrize("dtype", HALF)
def test_process_against_fp32(pq, bank, dtype, cls):
    from pqmf_b200 import _lib

    mod = bank(cls, 100, 16)
    delay = 1 if cls == "CachedPQMF" else 0
    x = signal((400, 1, 1 << 16), dtype, seed=31)
    b, t = x.shape[0], x.shape[-1]
    hk = mod.hk.float().contiguous()
    y_rc, out_rc = torch.empty(b, 16, t // 16, dtype=dtype, device="cuda"), torch.empty_like(x)
    rc = _lib.cabi.pqmf_roundtrip_x(x.data_ptr(), y_rc.data_ptr(), out_rc.data_ptr(), hk.data_ptr(), tables_ptr(mod), b, t, t // 16, 16,
                                    hk.shape[1], delay, mod._flags, dtype_code(dtype), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert rc == 0
    out, y = mod.process(x)
    y_ref = mod(x.float()).to(dtype)
    assert same_bits(y, y_ref)
    assert same_bits(out, mod.inverse(y_ref.float()).to(dtype))  # the synthesis reads the rounded sub-bands


@pytest.mark.parametrize("cls", CLASSES)
@pytest.mark.parametrize("dtype", HALF)
def test_reconstruct_against_fp32(pq, bank, dtype, cls):
    """1000 rows of 2^16 samples: three chunks of the default 96 MiB scratch (384, 384, 232 rows), the last one still native."""
    from pqmf_b200 import _lib

    mod = bank(cls, 100, 16)
    delay = 1 if cls == "CachedPQMF" else 0
    x = signal((1000, 1, 1 << 16), dtype, seed=32)
    b, t = x.shape[0], x.shape[-1]
    hk = mod.hk.float().contiguous()
    nbytes = _lib.cabi.pqmf_reconstruct_scratch_bytes(b, t, t // 16, 16)
    scratch = torch.empty(nbytes // 4, device="cuda")
    out_rc = torch.empty_like(x)
    rc = _lib.cabi.pqmf_reconstruct_x(x.data_ptr(), out_rc.data_ptr(), scratch.data_ptr(), nbytes, hk.data_ptr(), tables_ptr(mod), b, t,
                                      t // 16, 16, hk.shape[1], delay, mod._flags, dtype_code(dtype), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert rc == 0
    y_ref = mod(x.float()).to(dtype)
    assert same_bits(mod.reconstruct(x), mod.inverse(y_ref.float()).to(dtype))


# ---------------------------------------------------------------- 5. autograd in the steady state
@pytest.mark.parametrize("dtype", HALF)
@pytest.mark.parametrize("direction", ["analysis", "synthesis"])
@pytest.mark.parametrize("mag", [1e-2, 1e3])
def test_autograd_steady_state(bank, dtype, direction, mag):
    mod = bank("PQMF", 100, 16)
    shape = steady_shape(16)
    if direction == "analysis":
        inp = signal(shape, dtype, seed=41)
        fn = mod.forward
        g_shape = (shape[0], 16, shape[-1] // 16)
    else:
        inp = mod(signal(shape, dtype, seed=42))
        fn = mod.inverse
        g_shape = shape
    gen = torch.Generator(device="cuda").manual_seed(43)
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


# ---------------------------------------------------------------- 6. 64-bit offsets
@pytest.mark.parametrize("dtype,rows", [(torch.bfloat16, 4097), (torch.float32, 2049)])
def test_64_bit_offsets(pq, bank, dtype, rows):
    """Rows of 2^19 samples at n_band 16: bf16 with more than 2^31 elements, float32 with more than 2^32 bytes.  The last row
    starts beyond either limit.  About 13 GB of device memory."""
    free, _ = torch.cuda.mem_get_info()
    if free < 20 * 2 ** 30:
        pytest.skip(f"needs 20 GB of free device memory, {free / 2 ** 30:.1f} GB free")
    mod = bank("PQMF", 100, 16)
    t = 1 << 19
    x = torch.empty(rows, 1, t, dtype=dtype, device="cuda")
    for r0 in range(0, rows, 512):
        x[r0:r0 + 512] = signal((min(512, rows - r0), 1, t), dtype, seed=r0)
    assert x.numel() > 2 ** 31 if dtype == torch.bfloat16 else x.numel() * 4 > 2 ** 32
    ends = torch.tensor([0, 1, rows - 2, rows - 1], device="cuda")
    x_ends = x[ends].contiguous()
    y = mod(x)
    if dtype != torch.float32:
        assert rc_analysis(mod, x, t // 16) == 0
    del x
    out = mod.inverse(y)
    if dtype != torch.float32:
        assert rc_synthesis(mod, y, 0) == 0
    # two rows are 128 tiles: the same kernels run them as a separate batch
    for k in (slice(0, 2), slice(2, 4)):
        y_sep = mod(x_ends[k])
        assert same_bits(y_sep, y[ends[k]])
        assert same_bits(mod.inverse(y_sep), out[ends[k]])
    oracle_rows(mod, x_ends, y[ends], out[ends], 0, rows=(3,))
    del y, out
    torch.cuda.empty_cache()
