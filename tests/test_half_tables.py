"""Module casts and the fast-path tables (CPU only): ``_tables`` holds the bank's fp16 images as packed bits in a float32 buffer, so a
numeric cast of that buffer would corrupt them.  After any dtype cast it must be float32 and equal to the tables of the bank as it
now is."""
import pytest
import torch


@pytest.fixture(scope="module")
def pq():
    import pqmf_b200

    return pqmf_b200


def _assert_tables_follow_bank(mod, lib):
    expected, _, _ = lib.build_tables(mod.hk.float(), mod.h.float())
    assert mod._tables.dtype == torch.float32
    assert torch.equal(mod._tables.view(torch.int32), expected.view(torch.int32))


@pytest.mark.parametrize("n_band", [4, 16, 32])
@pytest.mark.parametrize("cast", ["half", "bfloat16", "half_float", "double", "bfloat16_half"])
@pytest.mark.parametrize("cls", ["PQMF", "CachedPQMF"])
def test_tables_rebuilt_after_dtype_cast(pq, cls, cast, n_band):
    from pqmf_b200 import _lib

    mod = getattr(pq, cls)(100, n_band)
    if cast == "half":
        mod = mod.half()
        want = torch.float16
    elif cast == "bfloat16":
        mod = mod.to(torch.bfloat16)
        want = torch.bfloat16
    elif cast == "half_float":
        mod = mod.half().float()
        want = torch.float32
    elif cast == "bfloat16_half":
        mod = mod.to(torch.bfloat16).half()
        want = torch.float16
    else:
        mod = mod.double()
        want = torch.float64
    assert mod.hk.dtype == want and mod.h.dtype == want
    _assert_tables_follow_bank(mod, _lib)
    if cls == "CachedPQMF":  # the streaming state is fp32 whatever the bank's dtype
        assert mod._x_state.dtype == torch.float32 and mod._s_state.dtype == torch.float32


def test_half_float_round_trip_equals_a_fresh_module_with_the_rounded_bank(pq):
    from pqmf_b200 import _lib

    mod = pq.PQMF(100, 16).half().float()
    fresh = pq.PQMF(100, 16)
    with torch.no_grad():
        fresh.hk.copy_(mod.hk)
        fresh.h.copy_(mod.h)
    fresh.refresh_tables()
    assert torch.equal(mod._tables.view(torch.int32), fresh._tables.view(torch.int32))
    assert mod._flags == fresh._flags
    _assert_tables_follow_bank(mod, _lib)


def test_fp32_module_and_state_dict_unchanged_by_casts(pq):
    mod = pq.CachedPQMF(100, 16)
    keys = list(mod.state_dict().keys())
    tables, flags = mod._tables.clone(), mod._flags
    mod.float()  # a no-op cast keeps the tables bit-equal without a rebuild
    assert torch.equal(mod._tables.view(torch.int32), tables.view(torch.int32)) and mod._flags == flags
    half = pq.CachedPQMF(100, 16).to(torch.bfloat16)
    assert list(half.state_dict().keys()) == keys
    assert half.state_dict()["hk"].dtype == torch.bfloat16
