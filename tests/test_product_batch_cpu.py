"""Batched independent products (sipp_inner_product_batch and friends) without a GPU: the host plan that cuts the segments into
accumulator groups and line-table chunks, every argument error (all of them are found before the device is touched), and the
loud failure of a valid call on a machine without a device."""
import ctypes
import random

import pytest

LINES_BYTES_PER_PAIR = 91 * 80 * 4
BUDGET_PAIRS = (16 << 30) // LINES_BYTES_PER_PAIR   # the 16 GB line-table budget of one call, in pairs


@pytest.fixture(scope="module")
def lib():
    from sipp_b200 import _lib
    return _lib.load()


def offsets_of(lengths):
    offs = [0]
    for length in lengths:
        offs.append(offs[-1] + length)
    return offs


def plan(lib, lengths, kpg_max, chunk_pairs):
    offs = offsets_of(lengths)
    arr = (ctypes.c_size_t * len(offs))(*offs)
    kpg = ctypes.c_int(0)
    g = lib.sipp_test_product_plan(arr, len(lengths), kpg_max, chunk_pairs, None, 0, ctypes.byref(kpg))
    assert g >= 0
    out = (ctypes.c_size_t * max(1, 4 * g))()
    assert lib.sipp_test_product_plan(arr, len(lengths), kpg_max, chunk_pairs, out, 4 * g, None) == g
    return kpg.value, [tuple(out[4 * i:4 * i + 4]) for i in range(g)], offs


def check_plan(kpg, groups, offs, kpg_max, chunk_pairs):
    cap = min(chunk_pairs, BUDGET_PAIRS) if chunk_pairs else BUDGET_PAIRS
    assert 1 <= kpg <= max(1, kpg_max)
    pos = 0
    for first, pairs, seg, chunk in groups:
        assert first == pos and 1 <= pairs <= kpg                      # the groups partition the flat pair list in order
        assert offs[seg] <= first and first + pairs <= offs[seg + 1]    # ... and no group crosses a segment
        assert first // cap == chunk == (first + pairs - 1) // cap      # ... or a chunk
        pos += pairs
    assert pos == offs[-1]
    # greedy cuts: inside one segment and one chunk every group but the last is full
    for (f0, p0, s0, c0), (f1, p1, s1, c1) in zip(groups, groups[1:]):
        if (s0, c0) == (s1, c1):
            assert p0 == kpg
    # every non-empty segment has groups, and they are consecutive
    segs = [g[2] for g in groups]
    assert segs == sorted(segs)
    assert set(segs) == {j for j in range(len(offs) - 1) if offs[j + 1] > offs[j]}


RAGGED = [0, 1, 2, 3, 5, 7, 8, 31, 64, 100, 129, 0, 1500]


def _skewed(long_len, seed=5, count=4095):
    rng = random.Random(seed)
    return [long_len] + [rng.randrange(0, 65) for _ in range(count)]


@pytest.mark.parametrize("lengths", [RAGGED, [0, 0, 0], [1] * 1000, [128] * 4096, _skewed(1 << 16), [1 << 16]],
                         ids=["ragged", "all-empty", "unit", "uniform-4096x128", "skewed", "one-long"])
@pytest.mark.parametrize("kpg_max", [1, 32])
@pytest.mark.parametrize("chunk_pairs", [0, 1, 37, 100, 4096])
def test_plan_invariants(lib, lengths, kpg_max, chunk_pairs):
    kpg, groups, offs = plan(lib, lengths, kpg_max, chunk_pairs)
    check_plan(kpg, groups, offs, kpg_max, chunk_pairs)
    if kpg_max == 1:
        assert kpg == 1 and len(groups) == offs[-1]


def test_plan_choices(lib):
    """the cost model's choices on the shapes the measurements use, and the forced chunks really cut"""
    assert plan(lib, [128] * 4096, 32, 0)[0] == 32          # 16,384 groups of 32: three waves of 148 x 40 groups
    assert plan(lib, [1] * 65536, 32, 0)[0] == 1             # one pair per product: nothing to share
    assert plan(lib, [3] * 10, 32, 0)[0] == 1                # 10 products of 3 pairs fit one wave at kpg = 1
    assert plan(lib, [128] * 4096, 5, 0)[0] == 5             # kpg_max need not be a power of two, nor kpg
    assert plan(lib, [1 << 16], 32, 0)[0] == 12              # one wave of 5,462 groups, as sipp_inner_product on the same pairs
    kpg, groups, offs = plan(lib, [100, 100], 32, 37)
    assert {g[3] for g in groups} == {0, 1, 2, 3, 4, 5}      # 200 pairs in chunks of 37
    assert any(g[2] == 0 and g[3] == 2 for g in groups) and any(g[2] == 1 and g[3] == 2 for g in groups)  # a chunk shared by two segments
    kpg, groups, offs = plan(lib, [1 << 20], 32, 0)
    assert max(g[3] for g in groups) == (1 << 20) // BUDGET_PAIRS  # 2^20 pairs need two chunks of the 16 GB budget


def test_plan_hook_errors(lib):
    from sipp_b200 import _lib
    arr = (ctypes.c_size_t * 3)(0, 5, 3)
    assert lib.sipp_test_product_plan(arr, 2, 32, 0, None, 0, None) == _lib.ERR_ARG
    assert lib.sipp_test_product_plan(None, 2, 32, 0, None, 0, None) == _lib.ERR_ARG
    assert lib.sipp_test_product_plan(arr, 0, 32, 0, None, 0, None) == 0


def _offs(*v):
    return (ctypes.c_size_t * len(v))(*v)


def test_argument_errors(lib):
    """every argument error comes before the device is touched, so these hold with and without a GPU"""
    from sipp_b200 import _lib
    A, B, out = bytes(64 * 3), bytes(128 * 3), ctypes.create_string_buffer(384 * 2)
    ok = _offs(0, 1, 3)
    assert lib.sipp_inner_product_batch(A, 3, B, 2, ok, 2, out) == _lib.ERR_LENGTH
    assert lib.sipp_inner_product_batch(None, 3, B, 3, ok, 2, out) == _lib.ERR_ARG
    assert lib.sipp_inner_product_batch(A, 3, None, 3, ok, 2, out) == _lib.ERR_ARG
    assert lib.sipp_inner_product_batch(A, 3, B, 3, None, 2, out) == _lib.ERR_ARG
    assert lib.sipp_inner_product_batch(A, 3, B, 3, ok, 2, None) == _lib.ERR_ARG
    assert lib.sipp_inner_product_batch(A, 3, B, 3, _offs(1, 2, 3), 2, out) == _lib.ERR_ARG       # offsets[0] != 0
    assert lib.sipp_inner_product_batch(A, 3, B, 3, _offs(0, 2, 1, 3), 3, out) == _lib.ERR_ARG    # decreasing
    assert lib.sipp_inner_product_batch(A, 3, B, 3, _offs(0, 1, 2), 2, out) == _lib.ERR_ARG       # offsets[count] != a_len
    assert lib.sipp_inner_product_batch(A, 3, B, 3, _offs(0, 1, 4), 2, out) == _lib.ERR_ARG
    assert lib.sipp_inner_product_batch(A, 3, B, 3, ok, 0, out) == _lib.ERR_ARG                   # count == 0 with pairs
    for args in ((None, 1, ok, 2, 1), (1, None, ok, 2, 1), (1, 1, None, 2, 1), (1, 1, ok, 2, None)):
        assert lib.sipp_inner_product_batch_device(args[0], args[1], 3, args[2], args[3], args[4]) == _lib.ERR_ARG
    assert lib.sipp_inner_product_batch_device(1, 1, 3, _offs(0, 3, 2), 2, 1) == _lib.ERR_ARG
    assert lib.sipp_pairing_batch(None, B, 3, out) == _lib.ERR_ARG
    assert lib.sipp_pairing_batch(A, B, 3, None) == _lib.ERR_ARG


def test_python_argument_errors():
    import sipp_b200
    with pytest.raises(AssertionError):
        sipp_b200.inner_product_batch(bytes(64 * 3), bytes(128 * 2), [3])
    with pytest.raises(ValueError):
        sipp_b200.inner_product_batch(bytes(64 * 3), bytes(128 * 3), [1, 1])
    with pytest.raises(ValueError):
        sipp_b200.inner_product_batch(bytes(64 * 3), bytes(128 * 3), [4, -1])
    with pytest.raises(AssertionError):
        sipp_b200.pairing_batch(bytes(64 * 2), bytes(128 * 3))
    with pytest.raises(ValueError):
        sipp_b200.inner_product_batch_device(1, 1, 3, [2], 1)


def test_no_gpu_fails_loudly(lib):
    """a valid call without a device returns SIPP_ERR_CUDA like every compute entry point (count == 0 included)"""
    import sipp_b200
    from sipp_b200 import _lib
    if lib.sipp_device_count() > 0:
        pytest.skip("a GPU is present")
    out = ctypes.create_string_buffer(384 * 2)
    assert lib.sipp_inner_product_batch(bytes(64 * 3), 3, bytes(128 * 3), 3, _offs(0, 1, 3), 2, out) == _lib.ERR_CUDA
    assert out.raw == bytes(384 * 2)
    assert lib.sipp_inner_product_batch(b"", 0, b"", 0, _offs(0), 0, out) == _lib.ERR_CUDA
    assert lib.sipp_inner_product_batch_device(1, 1, 3, _offs(0, 3), 1, 1) == _lib.ERR_CUDA
    assert lib.sipp_pairing_batch(bytes(64), bytes(128), 1, out) == _lib.ERR_CUDA
    with pytest.raises(sipp_b200.SippError) as ei:
        sipp_b200.pairing_batch(bytes(64), bytes(128))
    assert ei.value.code == _lib.ERR_CUDA
