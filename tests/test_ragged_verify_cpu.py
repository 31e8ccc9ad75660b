"""Ragged batched verification (sipp_verify_native_batch_ragged) without a GPU: every argument error and its code (all of them come
before the device is touched, in the order of the ragged prover's checks), the loud failure of a valid call without a device, and
the Python wrapper's ValueErrors."""
import ctypes

import pytest


@pytest.fixture(scope="module")
def lib():
    from sipp_b200 import _lib
    return _lib.load()


def _offs(*o):
    return (ctypes.c_size_t * len(o))(*o)


A, B = bytes(64 * 6), bytes(128 * 6)
OK_OFFS = (0, 2, 6)                      # n = 2, 4: proofs of 3 and 5 elements
OK_POFFS = (0, 3, 8)


def call(lib, a=A, a_len=6, b=B, b_len=6, offs=OK_OFFS, count=2, proofs=bytes(384 * 8), poffs=OK_POFFS, results=True, sentinel=None):
    res = (ctypes.c_int * max(1, count))(*([sentinel if sentinel is not None else 0] * max(1, count)))
    fa, fb, fz = (ctypes.create_string_buffer(b"\x5a" * (k * 3), k * 3) for k in (64, 128, 384))
    rc = lib.sipp_verify_native_batch_ragged(a, a_len, b, b_len, None if offs is None else _offs(*offs), count, proofs,
                                             None if poffs is None else _offs(*poffs), res if results else None, fa, fb, fz)
    return rc, list(res), (fa.raw, fb.raw, fz.raw)


def test_offsets_errors(lib):
    """the offsets checks of the ragged prover, with the same codes"""
    from sipp_b200 import _lib
    assert call(lib, b_len=5)[0] == _lib.ERR_LENGTH
    assert call(lib, a=None)[0] == _lib.ERR_ARG
    assert call(lib, b=None)[0] == _lib.ERR_ARG
    assert call(lib, offs=None)[0] == _lib.ERR_ARG
    assert call(lib, proofs=None)[0] == _lib.ERR_ARG
    assert call(lib, count=0)[0] == _lib.ERR_ARG                                     # count == 0
    assert call(lib, offs=(1, 2, 6))[0] == _lib.ERR_ARG                              # offsets[0] != 0
    assert call(lib, offs=(0, 4, 2, 6), count=3, poffs=(0, 5, 8, 11))[0] == _lib.ERR_ARG   # decreasing
    assert call(lib, offs=(0, 2, 4))[0] == _lib.ERR_ARG                              # offsets[count] != a_len
    assert call(lib, offs=(0, 0, 2, 6), count=3, poffs=(0, 1, 4, 9))[0] == _lib.ERR_ARG   # an empty instance
    assert call(lib, offs=(0, 3, 6))[0] == _lib.ERR_ARG                              # not a power of two
    assert call(lib, offs=(0, 6), count=1, poffs=(0, 8))[0] == _lib.ERR_ARG
    big = 1 << 32                                                                    # more than 2^32 - 1 pairs (never read)
    assert call(lib, a_len=big, b_len=big, offs=(0, big), count=1, poffs=(0, 65))[0] == _lib.ERR_ARG
    # the length check comes first, the offsets checks before those of the proofs
    assert call(lib, b_len=5, results=False)[0] == _lib.ERR_LENGTH
    assert call(lib, offs=(0, 3, 6), poffs=(0, 0, 0))[0] == _lib.ERR_ARG               # not SIPP_ERR_SHORT_PROOF


def test_proof_offsets_and_results_errors(lib):
    from sipp_b200 import _lib
    assert call(lib, results=False)[0] == _lib.ERR_ARG                               # NULL results
    assert call(lib, poffs=None)[0] == _lib.ERR_ARG                                  # NULL proof_offsets
    assert call(lib, poffs=(1, 3, 8))[0] == _lib.ERR_ARG                             # proof_offsets[0] != 0
    assert call(lib, poffs=(0, 9, 8))[0] == _lib.ERR_ARG                             # decreasing
    assert call(lib, poffs=(0, 2, 8))[0] == _lib.ERR_SHORT_PROOF                     # proof 0: 2 < 3 elements
    assert call(lib, poffs=(0, 3, 7))[0] == _lib.ERR_SHORT_PROOF                     # proof 1: 4 < 5 elements
    assert call(lib, poffs=(0, 0, 5))[0] == _lib.ERR_SHORT_PROOF                     # an empty proof
    # an n = 1 instance reads one element (Z); a decreasing pair is an argument error before any length is compared
    assert call(lib, a_len=2, b_len=2, offs=(0, 1, 2), poffs=(0, 0, 1))[0] == _lib.ERR_SHORT_PROOF
    assert call(lib, poffs=(0, 2, 1))[0] == _lib.ERR_ARG


def test_errors_write_nothing(lib):
    """an argument error leaves results and the finals as they were"""
    from sipp_b200 import _lib
    for kw in ({"poffs": (0, 2, 8)}, {"offs": (0, 3, 6)}, {"b_len": 5}):
        rc, res, fin = call(lib, sentinel=77, **kw)
        assert rc != _lib.OK
        assert res == [77, 77]
        assert fin == (b"\x5a" * 192, b"\x5a" * 384, b"\x5a" * 1152)


def test_no_gpu_fails_loudly(lib):
    """a valid call without a device returns SIPP_ERR_CUDA and writes nothing; longer proofs are valid arguments"""
    import sipp_b200
    from sipp_b200 import _lib
    if lib.sipp_device_count() > 0:
        pytest.skip("a GPU is present")
    for poffs in (OK_POFFS, (0, 4, 12)):
        rc, res, fin = call(lib, poffs=poffs, proofs=bytes(384 * 12), sentinel=77)
        assert rc == _lib.ERR_CUDA
        assert res == [77, 77]
        assert fin == (b"\x5a" * 192, b"\x5a" * 384, b"\x5a" * 1152)
    with pytest.raises(sipp_b200.SippError) as ei:
        sipp_b200.sipp_verify_native_batch_ragged(A, B, [2, 4], [[bytes(384)] * 3, [bytes(384)] * 5])
    assert ei.value.code == _lib.ERR_CUDA


def test_python_argument_errors():
    import sipp_b200
    good = [[bytes(384)] * 3, [bytes(384)] * 5]
    for lengths in ([3, 3], [6], [0, 2, 4], [-2, 8], [2, 2]):                      # as sipp_prove_native_batch_ragged
        with pytest.raises(ValueError):
            sipp_b200.sipp_verify_native_batch_ragged(A, B, lengths, good)
    with pytest.raises(ValueError):
        sipp_b200.sipp_verify_native_batch_ragged(b"", b"", [], [])                # no instances
    with pytest.raises(ValueError):
        sipp_b200.sipp_verify_native_batch_ragged(A, B, [2, 4], good[:1])          # one proof per instance
    with pytest.raises(ValueError):
        sipp_b200.sipp_verify_native_batch_ragged(A, B, [2, 4], [bytes(384 * 3), bytes(384 * 5 - 1)])   # not whole Fq12
    with pytest.raises(AssertionError):
        sipp_b200.sipp_verify_native_batch_ragged(A, bytes(128 * 4), [2, 4], good)
