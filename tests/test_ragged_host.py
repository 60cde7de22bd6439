"""Ragged batches without a GPU: the micro-batch schedule of ``runtime.ragged_batches`` and the argument checks of the
``*_ragged`` C-ABI entry points (validation happens before any CUDA call)."""
import ctypes
import random

import pytest


def test_ragged_batches_partition_order_and_padding():
    from megatts2_hierspeechpp_b200.runtime import ragged_batches
    rng = random.Random(5)
    lengths = [rng.randint(100, 1000) for _ in range(256)]
    idx = list(range(0, 256, 2)) + list(range(1, 256, 2))
    out = ragged_batches(idx, lengths, max_batch=16, frame_multiple=50)
    flat = [i for ids, _ in out for i in ids]
    assert sorted(flat) == list(range(256))                           # a partition of the input
    assert [lengths[i] for i in flat] == sorted(lengths, reverse=True)  # longest first, consecutive runs
    for ids, Tp in out:
        assert 1 <= len(ids) <= 16
        assert Tp % 50 == 0 and Tp - 50 < max(lengths[i] for i in ids) <= Tp
    assert all(len(ids) == 16 for ids, _ in out[:-1])
    assert ragged_batches(idx, lengths, 16, 50) == out                  # deterministic
    assert ragged_batches(list(reversed(idx)), lengths, 16, 50) == out  # ties broken by index, not input order
    assert len({Tp for _, Tp in out}) <= 19                            # (1000 - 100) / 50 + 1 possible shapes
    assert ragged_batches([], lengths, 4) == []
    assert ragged_batches([3], [7, 7, 7, 51], 4, frame_multiple=1) == [([3], 51)]
    assert ragged_batches([0, 1, 2], [5, 9, 5], 2, frame_multiple=4) == [([1, 0], 12), ([2], 8)]
    with pytest.raises(ValueError):
        ragged_batches([0], [5], 0)


@pytest.fixture(scope="module")
def lib():
    from megatts2_hierspeechpp_b200 import _lib, build
    build.build()
    return _lib.load()


def test_ragged_symbols_reject_bad_arguments(lib):
    one = ctypes.c_void_p(16)
    rc = lib.hsv_act1d_snakebeta_ragged(None, None, None, None, one, 1, 16, 64, 0, 1.0, None)
    assert rc == -1 and b"null" in lib.hsv_last_error()
    rc = lib.hsv_pack_blk16_sum3_ragged(None, None, None, one, None, 1, 16, 64, 0, 1.0, None)
    assert rc == -1 and b"null" in lib.hsv_last_error()
    rc = lib.hsv_pack_blk16_sum3_ragged(one, None, one, one, one, 1, 16, 64, 0, 1.0, None)
    assert rc == -1 and b"x3 without x2" in lib.hsv_last_error()
    rc = lib.hsv_conv1d_direct_ragged(None, None, None, one, None, 1, 32, 1, 64, 64, 7, 1, 3, 0, None)
    assert rc == -1 and b"null" in lib.hsv_last_error()
    rc = lib.hsv_sr_pre_interp_ragged(None, None, None, one, one, None, 1, 32, 64, 96, None)
    assert rc == -1 and b"null" in lib.hsv_last_error()
    # lengths are supported on the conv_post shape only (Cout <= 4, k 7, d 1, 'same' padding)
    for cout, k, d, pad in ((8, 7, 1, 3), (1, 3, 1, 1), (1, 7, 2, 6)):
        rc = lib.hsv_conv1d_direct_ragged(one, one, None, one, one, 1, 32, cout, 64, 64, k, d, pad, 0, None)
        assert rc == -1 and b"valid lengths" in lib.hsv_last_error(), (cout, k, d, pad)


def test_forced_tensor_core_activation_takes_no_lengths(lib):
    one = ctypes.c_void_p(16)
    lib.hsv_set_act_variant(2)
    try:
        rc = lib.hsv_act1d_snakebeta_ragged(one, one, one, one, one, 1, 16, 1024, 1, 1.0, None)
        assert rc == -1 and b"tensor-core" in lib.hsv_last_error()
    finally:
        lib.hsv_set_act_variant(0)
