"""Ragged batched proving (sipp_prove_native_batch_ragged) without a GPU: every argument error (all of them come before the device is
touched), the loud failure of a valid call without a device, the host schedule of the lock-step rounds, and the slices of
shard_instances_ragged."""
import ctypes
import math
import random

import pytest

LINES_BYTES_PER_PAIR = 91 * 80 * 4
BUDGET_PAIRS = (16 << 30) // LINES_BYTES_PER_PAIR   # the 16 GB line-table budget of one call, in pairs
STRAUS_MIN, WIDE_FOLD_MAX = 16384, 256               # fold thresholds of the batched prover (defaults)


@pytest.fixture(scope="module")
def lib():
    from sipp_b200 import _lib
    return _lib.load()


@pytest.fixture
def options(lib):
    """every option this file sets is restored afterwards"""
    saved = {k: lib.sipp_get_option(k) for k in range(1, 19)}
    yield
    for k, v in saved.items():
        lib.sipp_set_option(k, v)


def _offs(*o):
    return (ctypes.c_size_t * len(o))(*o)


def offsets_of(lengths):
    offs = [0]
    for length in lengths:
        offs.append(offs[-1] + length)
    return offs


def schedule(lib, lengths):
    offs = offsets_of(lengths)
    arr = (ctypes.c_size_t * len(offs))(*offs)
    rounds = lib.sipp_test_ragged_schedule(arr, len(lengths), None, 0)
    assert rounds > 0
    out = (ctypes.c_longlong * (5 * rounds))()
    assert lib.sipp_test_ragged_schedule(arr, len(lengths), out, 5 * rounds) == rounds
    return [tuple(out[5 * r:5 * r + 5]) for r in range(rounds)]


def _shapes():
    rng = random.Random(7)
    mixed = [1 << k for k in range(11)]
    shuffled = list(mixed) * 3
    rng.shuffle(shuffled)
    return {
        "ascending": mixed,
        "descending": mixed[::-1],
        "shuffled_duplicates": shuffled,
        "ones": [1] * 9,
        "single": [4096],
        "big_among_small": [16] * 100 + [4096] + [16] * 155,
        "cycling": [1 << (2 + (j % 8)) for j in range(64)],
    }


@pytest.mark.parametrize("name", sorted(_shapes()))
def test_schedule_totals(lib, options, name):
    """pairs over the rounds = sum (3 n_j - 2), fold elements = sum (n_j - 1), active counts follow log2 n_j"""
    lengths = _shapes()[name]
    sch = schedule(lib, lengths)
    logs = [int(math.log2(n)) for n in lengths]
    assert len(sch) == max(logs) + 1
    assert sum(r[1] for r in sch) == sum(3 * n - 2 for n in lengths)
    assert sum(r[2] for r in sch) == sum(n - 1 for n in lengths)
    acts = [r[0] for r in sch]
    assert acts == sorted(acts, reverse=True)                       # the active set only shrinks
    for r, (act, pairs, elems, kernel, chunks) in enumerate(sch):
        assert act == sum(1 for lg in logs if lg >= r)
        if r == 0:
            assert (pairs, elems, kernel) == (sum(lengths), 0, -1)
        else:
            assert elems == sum(n >> r for n in lengths if n >= (1 << r)) and pairs == 2 * elems
            want = 2 if elems >= STRAUS_MIN else 1 if elems <= WIDE_FOLD_MAX + 512 else 0
            assert kernel == want
        assert chunks == (pairs + BUDGET_PAIRS - 1) // BUDGET_PAIRS


def test_schedule_fold_kernels_follow_options(lib, options):
    from sipp_b200 import _lib
    lengths = [128] * 512                                           # 32768, 16384, 8192, ... 512 elements
    assert [r[3] for r in schedule(lib, lengths)] == [-1, 2, 2, 0, 0, 0, 0, 1]
    lib.sipp_set_option(_lib.OPT_FOLD_STRAUS, 0)
    assert [r[3] for r in schedule(lib, lengths)] == [-1, 0, 0, 0, 0, 0, 0, 1]
    lengths = [128] * 75                                            # 4800, 2400, 1200, 600, ... elements
    assert [r[3] for r in schedule(lib, lengths)] == [-1, 0, 0, 0, 1, 1, 1, 1]
    lib.sipp_set_option(_lib.OPT_WIDE_FOLD_MAX, 0)                  # the lane engine up to 512 elements only
    assert [r[3] for r in schedule(lib, lengths)] == [-1, 0, 0, 0, 0, 1, 1, 1]
    lib.sipp_set_option(_lib.OPT_WIDE_FOLD_MAX, 1 << 20)
    assert [r[3] for r in schedule(lib, lengths)] == [-1] + [1] * 7


@pytest.mark.parametrize("chunk", [37, 100, 1000])
def test_schedule_chunks(lib, options, chunk):
    """SIPP_OPT_PRODUCT_CHUNK_PAIRS cuts every round's products into chunks of at most that many pairs"""
    from sipp_b200 import _lib
    lib.sipp_set_option(_lib.OPT_PRODUCT_CHUNK_PAIRS, chunk)
    lengths = [64, 1, 8, 256, 2, 32, 4, 16]
    sch = schedule(lib, lengths)
    for act, pairs, elems, kernel, chunks in sch:
        assert chunks == (pairs + chunk - 1) // chunk
    lib.sipp_set_option(_lib.OPT_PRODUCT_CHUNK_PAIRS, 0)
    assert all(r[4] == 1 for r in schedule(lib, lengths))


def test_argument_errors(lib):
    """every argument error comes before the device is touched, so these hold with and without a GPU"""
    from sipp_b200 import _lib
    A, B, out = bytes(64 * 6), bytes(128 * 6), ctypes.create_string_buffer(384 * 8)
    ok = _offs(0, 2, 6)
    f = lib.sipp_prove_native_batch_ragged
    assert f(A, 6, B, 5, ok, 2, out) == _lib.ERR_LENGTH
    assert f(None, 6, B, 6, ok, 2, out) == _lib.ERR_ARG
    assert f(A, 6, None, 6, ok, 2, out) == _lib.ERR_ARG
    assert f(A, 6, B, 6, None, 2, out) == _lib.ERR_ARG
    assert f(A, 6, B, 6, ok, 2, None) == _lib.ERR_ARG
    assert f(A, 6, B, 6, ok, 0, out) == _lib.ERR_ARG                         # count == 0
    assert f(A, 6, B, 6, _offs(1, 2, 6), 2, out) == _lib.ERR_ARG             # offsets[0] != 0
    assert f(A, 6, B, 6, _offs(0, 4, 2, 6), 3, out) == _lib.ERR_ARG          # decreasing
    assert f(A, 6, B, 6, _offs(0, 2, 4), 2, out) == _lib.ERR_ARG             # offsets[count] != a_len
    assert f(A, 6, B, 6, _offs(0, 0, 2, 6), 3, out) == _lib.ERR_ARG          # an empty instance
    assert f(A, 6, B, 6, _offs(0, 3, 6), 2, out) == _lib.ERR_ARG             # not a power of two
    assert f(A, 6, B, 6, _offs(0, 6), 1, out) == _lib.ERR_ARG
    big = 1 << 32                                                            # more than 2^32 - 1 pairs (never read)
    assert f(A, big, B, big, _offs(0, big), 1, out) == _lib.ERR_ARG
    g = lib.sipp_prove_native_batch_ragged_device
    for args in ((None, 1, ok, 1), (1, None, ok, 1), (1, 1, None, 1), (1, 1, ok, None)):
        assert g(args[0], args[1], 6, args[2], 2, args[3]) == _lib.ERR_ARG
    assert g(1, 1, 6, _offs(0, 3, 6), 2, 1) == _lib.ERR_ARG
    assert g(1, 1, 6, ok, 0, 1) == _lib.ERR_ARG
    assert g(1, 1, big, _offs(0, big), 1, 1) == _lib.ERR_ARG
    assert lib.sipp_test_ragged_schedule(_offs(0, 3, 6), 2, None, 0) == _lib.ERR_ARG
    assert lib.sipp_test_ragged_schedule(None, 2, None, 0) == _lib.ERR_ARG


def test_python_argument_errors():
    import sipp_b200
    A, B = bytes(64 * 6), bytes(128 * 6)
    for lengths in ([3, 3], [6], [0, 2, 4], [-2, 8], [2, 2]):
        with pytest.raises(ValueError):
            sipp_b200.sipp_prove_native_batch_ragged(A, B, lengths)
    with pytest.raises(AssertionError):
        sipp_b200.sipp_prove_native_batch_ragged(A, bytes(128 * 4), [2, 4])
    with pytest.raises(ValueError):
        sipp_b200.sipp_prove_native_batch_ragged_device(1, 1, 6, [3, 3], 1)


def test_no_gpu_fails_loudly(lib):
    """a valid call without a device returns SIPP_ERR_CUDA and writes nothing"""
    import sipp_b200
    from sipp_b200 import _lib
    if lib.sipp_device_count() > 0:
        pytest.skip("a GPU is present")
    out = ctypes.create_string_buffer(384 * 4)
    assert lib.sipp_prove_native_batch_ragged(bytes(64 * 3), 3, bytes(128 * 3), 3, _offs(0, 1, 3), 2, out) == _lib.ERR_CUDA
    assert out.raw == bytes(384 * 4)
    assert lib.sipp_prove_native_batch_ragged_device(1, 1, 3, _offs(0, 2, 3), 2, 1) == _lib.ERR_CUDA
    with pytest.raises(sipp_b200.SippError) as ei:
        sipp_b200.sipp_prove_native_batch_ragged(bytes(64 * 3), bytes(128 * 3), [1, 2])
    assert ei.value.code == _lib.ERR_CUDA


@pytest.mark.parametrize("world", [1, 2, 3, 4, 8])
def test_shard_instances_ragged(world):
    """contiguous slices that cover every instance once, balanced by sum (3 n_j - 2)"""
    from sipp_b200.sharded import shard_instances_ragged
    rng = random.Random(world)
    for lengths in ([1 << rng.randrange(0, 11) for _ in range(300)], [4096] + [16] * 4095, [128] * 4096, [2, 1024, 4, 8]):
        cost = [3 * n - 2 for n in lengths]
        slices = [shard_instances_ragged(lengths, g, world) for g in range(world)]
        assert slices[0][0] == 0 and slices[-1][1] == len(lengths)
        for (lo, hi), (lo2, _) in zip(slices, slices[1:]):
            assert lo <= hi == lo2
        loads = [sum(cost[lo:hi]) for lo, hi in slices]
        ideal = sum(cost) / world
        for lo, hi in slices:   # a slice misses its share by at most the largest instance at each end
            assert abs(sum(cost[lo:hi]) - ideal) <= 2 * max(cost)
        if lengths == [128] * 4096:
            assert max(loads) - min(loads) <= 2 * cost[0]
