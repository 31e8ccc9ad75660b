"""Batched multi-exponentiations in GT (sipp_gt_msm_batch and its _device form) without a GPU: every argument error and its order, the
host form's encoding refusals before the device is touched, the loud failure of a valid call without a device, the per-segment plan
(path by length, window bits from the cost model), the forcing hook's refusals and the Python wrappers' ValueErrors."""
import ctypes

import pytest

P = 0x30644E72E131A029B85045B68181585D97816A916871CA8D3C208C16D87CFD47
R = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
FAKE = 0x7f0000001000   # a device address that is never read: every call below stops before the device is touched
SHORT_BELOW = 512        # segments shorter than this take the short path (include/sipp_b200.h)
ENTRIES = ("sipp_gt_msm_batch", "sipp_gt_msm_batch_device")


def le(v): return v.to_bytes(32, "little")


@pytest.fixture(scope="module")
def lib():
    from sipp_b200 import _lib
    return _lib.load()


def _szt(*o):
    return (ctypes.c_size_t * len(o))(*o)


def call(lib, name, elems=FAKE, scalars=FAKE, n=5, offs=(0, 2, 5), count=2, out=FAKE):
    if not name.endswith("_device"):  # valid host buffers unless the test passes None: the encoding checks read them
        elems = bytes(384 * n) if elems == FAKE else elems
        scalars = bytes(32 * n) if scalars == FAKE else scalars
        out = ctypes.create_string_buffer(max(1, 384 * count)) if out == FAKE else out
    return getattr(lib, name)(elems, scalars, n, None if offs is None else _szt(*offs), count, out)


@pytest.mark.parametrize("name", ENTRIES)
def test_argument_errors(lib, name):
    """the offsets rules of sipp_inner_product_batch, NULL pointers, count == 0 with elements, more than 2^32 - 1 elements: SIPP_ERR_ARG"""
    from sipp_b200 import _lib
    assert call(lib, name, elems=None) == _lib.ERR_ARG
    assert call(lib, name, scalars=None) == _lib.ERR_ARG
    assert call(lib, name, out=None) == _lib.ERR_ARG
    assert call(lib, name, offs=None) == _lib.ERR_ARG
    assert call(lib, name, offs=(1, 2, 5)) == _lib.ERR_ARG                     # offsets[0] != 0
    assert call(lib, name, offs=(0, 4, 2, 5), count=3) == _lib.ERR_ARG         # decreasing
    assert call(lib, name, offs=(0, 2, 4)) == _lib.ERR_ARG                     # offsets[count] != n
    assert call(lib, name, n=3, offs=(0,), count=0) == _lib.ERR_ARG            # count == 0 with elements
    if name.endswith("_device"):                                               # more than 2^32 - 1 elements (never read)
        big = 1 << 32
        assert call(lib, name, n=big, offs=(0, big), count=1) == _lib.ERR_ARG
        assert "2^32" in lib.sipp_last_error().decode()
    # the order: the NULL pointers before the offsets
    assert call(lib, name, elems=None, offs=(1, 2, 5)) == _lib.ERR_ARG
    assert "null" in lib.sipp_last_error().decode()


def test_host_encoding_refused_before_the_device(lib):
    """host form: a scalar >= r, then a coordinate >= p, give SIPP_ERR_ENCODING without a device, whatever the option values"""
    from sipp_b200 import _lib
    name = ENTRIES[0]
    for k in (R, R + 1, 2**256 - 1):
        assert call(lib, name, scalars=le(3) * 4 + le(k)) == _lib.ERR_ENCODING
        assert "r" in lib.sipp_last_error().decode()
    for slot in (0, 5, 11):  # the first, a middle and the last coordinate of an element
        g = bytearray(384 * 5)
        g[384 * 2 + 32 * slot:384 * 2 + 32 * slot + 32] = le(P)
        assert call(lib, name, elems=bytes(g), scalars=le(1) * 5) == _lib.ERR_ENCODING
        assert "p" in lib.sipp_last_error().decode()
    # p - 1 is canonical: the call gets as far as the device
    g = bytearray(384 * 5)
    g[0:32] = le(P - 1)
    if lib.sipp_device_count() == 0:
        assert call(lib, name, elems=bytes(g), scalars=le(R - 1) * 5) == _lib.ERR_CUDA
    # the scalar check comes first
    g[384 * 4:384 * 4 + 32] = le(P)
    assert call(lib, name, elems=bytes(g), scalars=le(R) * 5) == _lib.ERR_ENCODING
    assert "scalar" in lib.sipp_last_error().decode()


def test_no_gpu_fails_loudly(lib):
    """valid calls without a device return SIPP_ERR_CUDA, count == 0 included (as sipp_g1_msm_batch)"""
    import sipp_b200
    from sipp_b200 import _lib
    if lib.sipp_device_count() > 0:
        pytest.skip("a GPU is present")
    for name in ENTRIES:
        assert call(lib, name) == _lib.ERR_CUDA
        assert call(lib, name, n=0, offs=(0,), count=0) == _lib.ERR_CUDA
        assert call(lib, name, n=5, offs=(0, 0, 5, 5), count=3) == _lib.ERR_CUDA   # empty segments are valid
    # device buffers need only be 4-byte aligned
    assert call(lib, ENTRIES[1], elems=FAKE + 4, scalars=FAKE + 4, out=FAKE + 8) == _lib.ERR_CUDA
    with pytest.raises(sipp_b200.SippError) as ei:
        sipp_b200.gt_msm_batch_device(FAKE, FAKE, 5, [2, 3], FAKE)
    assert ei.value.code == _lib.ERR_CUDA
    with pytest.raises(sipp_b200.SippError) as ei:
        sipp_b200.gt_msm_batch([bytes(384)] * 2, [le(1)] * 2, [2])
    assert ei.value.code == _lib.ERR_CUDA


def test_python_argument_errors():
    import sipp_b200
    fn = sipp_b200.gt_msm_batch
    with pytest.raises(ValueError):
        fn(bytes(384 * 3), bytes(32 * 2), [3])            # elements / scalars
    with pytest.raises(ValueError):
        fn(bytes(384 * 3), bytes(32 * 3), [1, 1])         # lengths
    with pytest.raises(ValueError):
        fn(bytes(384 * 3), bytes(32 * 3), [4, -1])        # negative length
    with pytest.raises(ValueError):
        fn(bytes(384 * 3 + 1), bytes(32 * 3), [3])        # not whole elements
    with pytest.raises(ValueError):
        sipp_b200.gt_msm_batch_device(FAKE, FAKE, 5, [2, 2], FAKE)


def _window_bits(length):
    """the cost model of msm.cu: the c in 2..16 minimising W (len + 2 2^c) + c W Fq12 products, W = ceil(254 / c) (smallest c on ties)"""
    return min((-(-254 // c) * (length + 2 * 2 ** c) + c * -(-254 // c), c) for c in range(2, 17))[1]


def test_plan_thresholds(lib):
    """the short path below SHORT_BELOW elements (and for empty segments), Pippenger from there on, with the cost model's window size"""
    from sipp_b200 import _lib
    T = SHORT_BELOW
    lengths = [0, 1, 2, 15, 25, 300, T - 1, T, T + 1, 0, 1000, 4096, 1 << 16, 1 << 20, 0]
    offs = [0]
    for length in lengths:
        offs.append(offs[-1] + length)
    out = (ctypes.c_int * (2 * len(lengths)))()
    assert lib.sipp_test_gt_msm_plan(_szt(*offs), len(lengths), out, 2 * len(lengths)) == len(lengths)
    for j, length in enumerate(lengths):
        if length < T:
            assert (out[2 * j], out[2 * j + 1]) == (0, 0), length
        else:
            assert (out[2 * j], out[2 * j + 1]) == (1, _window_bits(length)), length
    # pinned points of the model: c grows with the length
    assert [_window_bits(n) for n in (512, 1000, 1 << 12, 1 << 16, 1 << 20)] == [6, 7, 8, 12, 16]
    # a short out buffer is not written
    short = (ctypes.c_int * 2)(-7, -7)
    assert lib.sipp_test_gt_msm_plan(_szt(*offs), len(lengths), short, 2) == len(lengths)
    assert list(short) == [-7, -7]
    # the entry points' offsets checks
    assert lib.sipp_test_gt_msm_plan(_szt(1, 2), 1, out, 2) == _lib.ERR_ARG
    assert lib.sipp_test_gt_msm_plan(_szt(0, 2, 1), 2, out, 4) == _lib.ERR_ARG
    assert lib.sipp_test_gt_msm_plan(_szt(0, 1 << 32), 1, out, 2) == _lib.ERR_ARG
    assert lib.sipp_test_gt_msm_plan(None, 1, out, 2) == _lib.ERR_ARG
    assert lib.sipp_test_gt_msm_plan(_szt(0), 0, out, 0) == 0


def test_forced_path_hook_arguments(lib):
    """sipp_test_gt_msm_batch_device: the path (c = 0 or 2 .. 16), then the device form's checks, all before the device"""
    from sipp_b200 import _lib
    f = lib.sipp_test_gt_msm_batch_device
    offs = _szt(0, 2, 5)
    for c in (1, 17, -1, 32):
        assert f(c, FAKE, FAKE, 5, offs, 2, FAKE) == _lib.ERR_ARG, c
        assert "c must" in lib.sipp_last_error().decode()
    assert f(0, None, FAKE, 5, offs, 2, FAKE) == _lib.ERR_ARG
    assert f(5, FAKE, FAKE, 5, _szt(1, 2, 5), 2, FAKE) == _lib.ERR_ARG
    assert f(2, FAKE, FAKE, 3, _szt(0), 0, FAKE) == _lib.ERR_ARG
    if lib.sipp_device_count() == 0:
        for c in (0, 2, 5, 16):
            assert f(c, FAKE, FAKE, 5, offs, 2, FAKE) == _lib.ERR_CUDA
